"""Every kernel variant of the direct `LHS \\ RHS` path (diffopt_b200_kkt_solve_csc, QuadraticProgram.jl:486-492) against
LAPACK / SuperLU, with the kernel that ran checked by name.

The host picks kernels from the shape alone, so each test builds a matrix whose shape lands in one variant and asserts,
through `torch.profiler`, that the variant ran:
  * one-CTA LU (`dense_lu_solve_kernel`) for N <= 128;
  * blocked LU (kkt_dense.cu) for N <= 1024 or a density of at least 2 %: each panel of height mr = N - k0 goes to
    `bl_panel_reg_kernel<32>` (mr <= 512), `bl_panel_reg_kernel<16>` (mr <= 1024), `bl_panel_kernel` staged in shared
    memory (kb narrowed to 16 while the panel fits the opt-in) or `bl_panel_kernel` in place in global memory (beyond);
  * multifrontal LU (sparse_mf.cu) otherwise: factor kernels `mf_factor_kernel<256|512|1024>` / `mf_factor_big_kernel`
    by front size, and the leaf / tiled / global `<true>` forward and backward sweeps.

Accuracy, for every system: relative forward error <= 1e-8 per column against LAPACK (SuperLU for the sparse route) on
well-conditioned matrices, and a normwise backward error ||r - K x||inf / (||K||inf ||x||inf + ||r||inf) per column, the
residual summed in long double, of at most 10x the backward error of LAPACK's own solution plus 1e-15: that bound
follows the system, and a wrong interchange or stride shows in it even where the forward error hides it."""
import re

import numpy as np
import pytest
import scipy.linalg as sl
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

import bench_data
import diffopt_b200
from oracle import qp as oqp

pytestmark = pytest.mark.gpu
RTOL_DIRECT = 1e-8
BL_NB = 32                 # block width of the blocked LU (kkt_dense.cu)
DENSE_MAX = 1024           # below this order every matrix takes a dense route (kkt_dense.cu, DIFFOPT_B200_DENSE_MAX)
MF_LEAF = 32               # vertices per leaf of the nested dissection (sparse_mf.cu)
MF_NRHS = (1, 64, 65, 128, 129, 257)   # across the 64-column tiles of the sweeps and the 128-column tiles of the leaves


@pytest.fixture(scope="module")
def ctx():
    return diffopt_b200.Context(0)


@pytest.fixture(scope="module")
def lsq():
    return diffopt_b200.submodule("lsqr")


@pytest.fixture(scope="module")
def optin():
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


# ---- which kernels ran ------------------------------------------------------------------------------------------------
def kernels_run(fn):
    """(names of the CUDA kernels `fn` launched, fn's result).  Fails, rather than passes every name check vacuously,
    when the profiler records no kernel at all."""
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


DENSE_ONE_CTA = r"\bdense_lu_solve_kernel\b"
BL_REG32, BL_REG16, BL_PANEL = r"\bbl_panel_reg_kernel<32>", r"\bbl_panel_reg_kernel<16>", r"\bbl_panel_kernel\b"
BL_OTHERS = (r"\bbl_swap_trsm_kernel\b", r"\bbl_gemm_kernel\b", r"\bbl_back_diag_kernel\b")
MF_ANY = r"\bmf_factor_(big_)?kernel\b"


# ---- accuracy -----------------------------------------------------------------------------------------------------------
def _matvec_ld(A, X):
    """A @ X summed in long double (A dense or sparse, X float64)."""
    if not sp.issparse(A):
        return np.asarray(A, dtype=np.longdouble) @ X.astype(np.longdouble)
    A = sp.csr_matrix(A)
    A.sort_indices()
    out = np.zeros(X.shape, np.longdouble)
    nonempty = np.diff(A.indptr) > 0
    starts = A.indptr[:-1][nonempty]
    vals = A.data.astype(np.longdouble)
    for c0 in range(0, X.shape[1], 32):
        prod = vals[:, None] * X[A.indices, c0:c0 + 32].astype(np.longdouble)
        out[nonempty, c0:c0 + 32] = np.add.reduceat(prod, starts, axis=0)
    return out


def backward_error(A, R, X):
    """Normwise backward error of every column of X as a solution of A X = R (residual in long double)."""
    res = np.abs(R.astype(np.longdouble) - _matvec_ld(A, X)).max(axis=0)
    norm_a = abs(A).sum(axis=1).max() if sp.issparse(A) else np.abs(A).sum(axis=1).max()
    return (res / (np.longdouble(norm_a) * np.abs(X).max(axis=0) + np.abs(R).max(axis=0))).astype(np.float64)


def reference(A, R):
    """LAPACK's (dense A) or SuperLU's (sparse A) solution of A X = R and its backward error per column."""
    X = spla.splu(sp.csc_matrix(A)).solve(R) if sp.issparse(A) else sl.lu_solve(sl.lu_factor(A), R)
    return X, backward_error(A, R, X)


def check_solution(A, R, X, ref=None, backward=True):
    """X solves A X = R as well as the reference does: forward error <= 1e-8 per column, backward error <= 10x the
    reference's + 1e-15.  `ref` = (X_ref, be_ref) for the leading columns of a larger reference solve."""
    Xr, be_ref = reference(A, R) if ref is None else ref
    Xr, be_ref = Xr[:, :X.shape[1]], be_ref[:X.shape[1]]
    assert np.isfinite(X).all()
    fwd = np.linalg.norm(X - Xr, axis=0) / np.linalg.norm(Xr, axis=0)
    assert fwd.max() <= RTOL_DIRECT, (fwd.max(), int(fwd.argmax()))
    if backward:
        be = backward_error(A, R, X)
        bad = be > 10.0 * be_ref + 1e-15
        assert not bad.any(), (np.flatnonzero(bad)[:8], be[bad][:8], be_ref[bad][:8])


def solve(lsq, ctx, K, R, trans=False):
    return lsq.solve_csc(ctx, sp.csc_matrix(K), R, trans=trans)


# ---- matrices -----------------------------------------------------------------------------------------------------------
def dense_kkt(n, m, p, seed):
    """LHS of one dense QP (create_LHS_matrix, QuadraticProgram.jl:256-282), order n + m + p."""
    d = bench_data.qp_batch(1, n, m, p, n_active=min(n // 4, 200), seed0=seed)
    return oqp.create_lhs(d["z"][0], d["lam"][0], d["Q"][0], d["G"][0], d["h"][0], d["A"][0])


def sparse_random(N, density, seed):
    """Random nonsymmetric pattern of the given density plus a dominant diagonal (well conditioned)."""
    rng = np.random.default_rng(seed)
    M = sp.random(N, N, density=density, random_state=np.random.RandomState(seed), format="csc",
                  data_rvs=lambda k: rng.standard_normal(k))
    return sp.csc_matrix(M + sp.diags(rng.uniform(2.0, 3.0, N) * rng.choice([-1, 1], N) * np.sqrt(density * N + 1)))


def cyclic_pivots(N, seed):
    """K = 10 C + E: C the cyclic shift with its ones at (N-1, 0), (0, 1), (1, 2), ..., E random +-1.  Partial pivoting
    takes the row C puts under the diagonal, which the previous interchange has just moved to the pivot row's old place:
    the same physical row index comes back for many consecutive columns (ipiv = N-1, N-1, ... at first)."""
    K = np.random.default_rng(seed).choice([-1.0, 1.0], (N, N))
    K[N - 1, 0] += 10.0
    K[np.arange(N - 1), np.arange(1, N)] += 10.0
    return K


def arrowhead(D, n_body=1000, chain=100, frac=0.3, seed=0):
    """D dense rows and columns over a sparse body of tridiagonal chains (length `chain`, nonsymmetric values).

    A vertex whose degree exceeds max(40, 10 sqrt(N)) is `dense` in the multifrontal analysis and eliminated last in one
    root front of order exactly D; every front below carries the dense vertices in its boundary.  The dense block is
    Gaussian (pivoting in the root front does real work), the couplings are small against the body's diagonal (no
    delayed pivots), so the front sizes, and the kernels they pick, follow from D."""
    rng = np.random.default_rng(seed)
    d = rng.uniform(1.0, 2.0, n_body) * rng.choice([-1, 1], n_body)
    lo, up = rng.standard_normal(n_body - 1) * 0.5, rng.standard_normal(n_body - 1) * 0.5
    lo[chain - 1::chain] = 0.0
    up[chain - 1::chain] = 0.0
    body = sp.diags([lo, d, up], [-1, 0, 1])
    rs = np.random.RandomState(seed)
    B = sp.random(n_body, D, density=frac, random_state=rs, data_rvs=lambda k: 0.1 * rng.standard_normal(k))
    C = sp.random(D, n_body, density=frac, random_state=rs, data_rvs=lambda k: 0.1 * rng.standard_normal(k))
    K = sp.bmat([[body, B], [C, sp.csr_matrix(rng.standard_normal((D, D)))]], format="csc")
    K.sort_indices()
    return K


def dense_vertex_count(K):
    """Vertices of the symmetrised pattern (diagonal excluded) above the analysis' dense-degree threshold."""
    N = K.shape[0]
    P = sp.csr_matrix(abs(K) + abs(K).T)
    P.setdiag(0)
    P.eliminate_zeros()
    return int((np.diff(P.indptr) > max(40.0, 10.0 * np.sqrt(N))).sum())


def _smem_factor(nf, k):
    """Dynamic shared memory of a front of order nf with k pivots in mf_factor_kernel (sparse_mf.cu)."""
    return (nf * (nf | 1) + k) * 8


def mf_factor_class(nf):
    """Factor kernel of a launch group whose largest front has order nf and nf pivots (a root front)."""
    smem = _smem_factor(nf, nf)
    if smem > 200 * 1024:
        return "big"
    return 1024 if smem > 100 * 1024 else 512 if smem > 50 * 1024 else 256


# (D, factor kernels, forward/backward sweeps that must run, sweeps that must not): see arrowhead().  The root front
# (order D, no boundary) decides the factor kernel of the top level; the leaves (<= 32 pivots plus the D dense rows in
# their boundary) and the chain separators (a few pivots) run beside it.
# The plain shared-memory sweeps (`mf_forward_kernel<false>`, `mf_backward_kernel<false>`) are reached by no matrix: a
# launch group takes them only if it is neither a leaf group, nor tiled, nor factorised in global memory.  Not factorised
# in global memory means nf (nf | 1) + k <= 25600 doubles, so nf <= 159; at nf <= 159 the tiled sweeps need at most
# 8 (159 * 73 + 1) + 4 (2 * 159 + 160 + 8192) = 127544 bytes forward (less backward), under the 200 KiB cap, so the group is
# tiled unless the net-permutation kernel was skipped, which takes a front with more than 25600 pivots.
MF_CASES = [
    (40, [r"\bmf_factor_kernel<256>"], ["leaf", "tiled"], ["true", "false"]),
    (90, [r"\bmf_factor_kernel<512>", r"\bmf_factor_kernel<1024>"], ["leaf", "tiled"], ["true", "false"]),
    (120, [r"\bmf_factor_kernel<1024>"], ["leaf", "tiled"], ["true", "false"]),
    (170, [r"\bmf_factor_big_kernel\b"], ["tiled"], ["leaf", "true", "false"]),
    (300, [r"\bmf_factor_big_kernel\b"], ["true"], ["leaf", "tiled", "false"]),
]
MF_ROOT_CLASS = {40: 256, 90: 512, 120: 1024, 170: "big", 300: "big"}


def _sweep(kind, direction):
    return {"leaf": rf"\bmf_{direction}_leaf_kernel\b", "tiled": rf"\bmf_{direction}_tiled_kernel\b",
            "true": rf"\bmf_{direction}_kernel<true>", "false": rf"\bmf_{direction}_kernel<false>"}[kind]


# ---- blocked LU panel regimes ---------------------------------------------------------------------------------------------
def panel_plan(N, optin):
    """(k0, kb, regime) of every block of dense_blocked_lu_solve (kkt_dense.cu), the same `fits()` arithmetic: a panel of
    mr = N - k0 rows lives in registers up to 512 (32 columns) / 1024 rows (16 columns); beyond, it is staged in shared
    memory while it fits the opt-in (narrowed to 16 columns if that makes it fit) and worked on in place otherwise."""
    def fits(mr, w):
        return 8 * mr * w + 2048 <= optin
    plan, k0 = [], 0
    while k0 < N:
        mr = N - k0
        kb = min(BL_NB, mr)
        if not fits(mr, kb) and kb > 16 and fits(mr, 16):
            kb = 16
        if mr <= 512:
            regime = "reg32"
        elif mr <= 1024:
            kb, regime = min(16, kb), "reg16"
        else:
            regime = "staged" if fits(mr, kb) else "inplace"
        plan.append((k0, kb, regime))
        k0 += kb
    return plan


REGIMES = ("inplace", "staged", "reg16", "reg32")


def staged_max_rows(optin):
    """Tallest panel the staged regime takes (16 columns in shared memory)."""
    return (optin - 2048) // (8 * 16)


def all_regimes_order(optin):
    """An order whose factorisation passes through all four panel regimes: a few in-place blocks first."""
    return staged_max_rows(optin) + 6 * BL_NB


def first_block(plan, regime):
    return next((k0, kb) for k0, kb, r in plan if r == regime)


# ==== dense routes ==========================================================================================================
@pytest.mark.parametrize("n,m,p,expect", [(50, 50, 28, "one_cta"), (50, 50, 29, "blocked")])
def test_route_boundary_one_cta_and_blocked(ctx, lsq, n, m, p, expect):
    """N = 128 is the largest order of the one-CTA LU, N = 129 the smallest of the blocked LU."""
    K = dense_kkt(n, m, p, seed=5100 + p)
    R = np.random.default_rng(p).standard_normal((K.shape[0], 3))
    names, X = kernels_run(lambda: solve(lsq, ctx, K, R))
    assert ran(names, DENSE_ONE_CTA) == (expect == "one_cta"), names
    assert ran(names, BL_REG32) == (expect == "blocked"), names
    assert not ran(names, MF_ANY), names
    check_solution(K, R, X)


@pytest.mark.parametrize("N", [DENSE_MAX, DENSE_MAX + 1])
@pytest.mark.parametrize("density", [0.005, 0.05])
def test_route_boundary_blocked_and_multifrontal(ctx, lsq, N, density):
    """Below 2 % density a matrix takes the blocked LU up to N = 1024 and the multifrontal LU from N = 1025; at 5 % it
    stays on the blocked LU on both sides."""
    K = sparse_random(N, density, seed=N)
    assert (K.nnz >= 0.02 * N * N) == (density > 0.02)
    R = np.random.default_rng(N).standard_normal((N, 3))
    multifrontal = N > DENSE_MAX and density < 0.02
    for trans in (False, True):
        names, X = kernels_run(lambda: solve(lsq, ctx, K, R, trans))
        assert ran(names, MF_ANY) == multifrontal, names
        assert ran(names, BL_REG32) == (not multifrontal), names
        check_solution(sp.csc_matrix(K.T) if trans else K, R, X)


def test_one_cta_and_blocked_lu_agree(ctx, lsq, monkeypatch):
    """DIFFOPT_B200_DENSE_ONE_CTA sends an N = 300 system through the one-CTA LU instead of the blocked one: both answers
    pass the accuracy check and agree with each other to rounding."""
    K = dense_kkt(120, 120, 60, seed=5300)
    R = np.random.default_rng(3).standard_normal((K.shape[0], 5))
    for trans in (False, True):
        A = K.T if trans else K
        ref = reference(A, R)
        names_b, Xb = kernels_run(lambda: solve(lsq, ctx, K, R, trans))
        monkeypatch.setenv("DIFFOPT_B200_DENSE_ONE_CTA", "1")
        names_o, Xo = kernels_run(lambda: solve(lsq, ctx, K, R, trans))
        monkeypatch.delenv("DIFFOPT_B200_DENSE_ONE_CTA")
        assert ran(names_b, BL_REG32) and not ran(names_b, DENSE_ONE_CTA), names_b
        assert ran(names_o, DENSE_ONE_CTA) and not ran(names_o, BL_REG32), names_o
        check_solution(A, R, Xb, ref)
        check_solution(A, R, Xo, ref)
        assert (np.linalg.norm(Xb - Xo, axis=0) / np.linalg.norm(Xo, axis=0)).max() <= 1e-11


def test_blocked_and_multifrontal_lu_agree(ctx, lsq, monkeypatch):
    """DIFFOPT_B200_DENSE_MAX moves a sparse N = 1100 system from the multifrontal LU to the blocked LU: same answer."""
    K = sparse_random(1100, 0.005, seed=11)
    R = np.random.default_rng(11).standard_normal((1100, 4))
    for trans in (False, True):
        A = sp.csc_matrix(K.T) if trans else K
        ref = reference(A, R)
        names_m, Xm = kernels_run(lambda: solve(lsq, ctx, K, R, trans))
        monkeypatch.setenv("DIFFOPT_B200_DENSE_MAX", "2048")
        names_b, Xb = kernels_run(lambda: solve(lsq, ctx, K, R, trans))
        monkeypatch.delenv("DIFFOPT_B200_DENSE_MAX")
        assert ran(names_m, MF_ANY) and not ran(names_m, BL_REG32), names_m
        assert ran(names_b, BL_REG32) and not ran(names_b, MF_ANY), names_b
        check_solution(A, R, Xm, ref)
        check_solution(A, R, Xb, ref)
        assert (np.linalg.norm(Xb - Xm, axis=0) / np.linalg.norm(Xm, axis=0)).max() <= 1e-12


# ==== blocked LU: all panel regimes =========================================================================================
def _kkt_of_order(N, seed):
    p = N // 8
    n = (N - p) // 2
    return dense_kkt(n, N - p - n, p, seed)


@pytest.mark.parametrize("extra_rows", [0, 2200])
def test_blocked_lu_all_panel_regimes(ctx, lsq, optin, extra_rows):
    """A dense KKT matrix tall enough that one factorisation passes through all four panel regimes (in place, staged,
    registers with 16 and with 32 columns); with 2100 more rows the in-place panels have more than four rows per thread
    in the strided argmax (r += 1024).  Both orientations; nrhs = 129 puts the backward diagonal block on two CTAs."""
    N = all_regimes_order(optin) + extra_rows
    plan = panel_plan(N, optin)
    assert {r for _, _, r in plan} == set(REGIMES), plan
    if extra_rows:
        assert N > 4 * 1024
    K = _kkt_of_order(N, seed=5400 + extra_rows)
    assert K.shape == (N, N) and np.count_nonzero(K) >= 0.02 * N * N
    rng = np.random.default_rng(N)
    for nrhs in ((1, 3) if extra_rows else (1, 129)):   # (long-double residuals of 4000 x 129 take a minute on the host)
        R = rng.standard_normal((N, nrhs))
        for trans in (False, True):
            A = K.T if trans else K
            names, X = kernels_run(lambda: solve(lsq, ctx, K, R, trans))
            for pat in (BL_REG32, BL_REG16, BL_PANEL) + BL_OTHERS:
                assert ran(names, pat), (pat, names)
            assert not ran(names, DENSE_ONE_CTA) and not ran(names, MF_ANY), names
            check_solution(A, R, X)


def _repeats(piv, k0, kb):
    return len(set(piv[k0:k0 + kb].tolist())) < kb


def test_blocked_lu_repeated_pivot_rows(ctx, lsq, optin):
    """K = 10 C + E (cyclic_pivots): partial pivoting takes the same row index several times inside one block, in every
    panel regime -- the position table of the register panels and the interchange replay of bl_swap_trsm_kernel."""
    N = all_regimes_order(optin)
    K = cyclic_pivots(N, seed=7)
    _, piv = sl.lu_factor(K)
    plan = panel_plan(N, optin)
    for regime in REGIMES:   # the case cannot go stale: LAPACK's own pivots repeat inside a block of every regime
        blocks = [(k0, kb) for k0, kb, r in plan if r == regime]
        assert any(_repeats(piv, k0, kb) for k0, kb in blocks), regime
    assert {16, 32} <= {kb for k0, kb, _ in plan if _repeats(piv, k0, kb)}
    R = np.random.default_rng(7).standard_normal((N, 3))
    for trans in (False, True):
        names, X = kernels_run(lambda: solve(lsq, ctx, K, R, trans))
        for pat in (BL_REG32, BL_REG16, BL_PANEL, BL_OTHERS[0]):
            assert ran(names, pat), (pat, names)
        check_solution(K.T if trans else K, R, X)


def test_one_cta_lu_repeated_pivot_rows(ctx, lsq):
    K = cyclic_pivots(120, seed=8)
    _, piv = sl.lu_factor(K)
    assert _repeats(piv, 0, 32)
    R = np.random.default_rng(8).standard_normal((120, 3))
    for trans in (False, True):
        names, X = kernels_run(lambda: solve(lsq, ctx, K, R, trans))
        assert ran(names, DENSE_ONE_CTA), names
        check_solution(K.T if trans else K, R, X)


def _singular_info(lsq, ctx, K):
    R = np.ones((K.shape[0], 2))
    with pytest.raises(diffopt_b200.SingularException) as e:
        solve(lsq, ctx, K, R)
    return e.value.info


@pytest.mark.parametrize("regime", REGIMES + ("one_cta",))
@pytest.mark.parametrize("kind", ["column", "row"])
def test_zero_pivot_index_matches_lapack(ctx, lsq, optin, regime, kind):
    """An exactly zero column inside a panel of the given regime (or a zero row there): the index of the first zero
    pivot, the argument of SingularException, is LAPACK's dgetrf `info`."""
    if regime == "one_cta":
        N, (k0, kb) = 100, (40, 32)
    else:
        N = all_regimes_order(optin)
        k0, kb = first_block(panel_plan(N, optin), regime)
    K = np.random.default_rng(N + k0).standard_normal((N, N))
    j = k0 + kb // 2 + 1
    if kind == "column":
        K[:, j] = 0.0
    else:
        K[j, :] = 0.0
    _, _, info = sl.lapack.dgetrf(K)
    assert info > 0
    assert _singular_info(lsq, ctx, K) == info


# ==== multifrontal LU =======================================================================================================
@pytest.mark.parametrize("D,factor,sweeps,absent", MF_CASES, ids=[f"D{c[0]}" for c in MF_CASES])
def test_multifrontal_kernel_variants(ctx, lsq, D, factor, sweeps, absent):
    """Arrowheads whose root front has order D reach each factor kernel and each solve sweep (MF_CASES); both
    orientations against SuperLU, nrhs across the 64-column tiles of the sweeps and the 128-column tiles of the leaves.
    The plain shared-memory sweeps `mf_forward_kernel<false>` / `mf_backward_kernel<false>` run for no matrix: see
    MF_CASES."""
    K = arrowhead(D)
    N = K.shape[0]
    assert dense_vertex_count(K) == D
    R = np.random.default_rng(D).standard_normal((N, max(MF_NRHS)))
    for trans in (False, True):
        A = sp.csc_matrix(K.T) if trans else K
        ref = reference(A, R)
        names, F = kernels_run(lambda: lsq.SparseFactorization(ctx, K, trans=trans))
        assert F.stats["method"] == "multifrontal" and F.stats["delayed_pivot_retries"] == 0, F.stats
        assert D <= F.stats["max_front"] <= D + MF_LEAF + 2, F.stats
        for pat in factor:
            assert ran(names, pat), (pat, names)
        for nrhs in MF_NRHS:
            if nrhs == max(MF_NRHS):
                names, X = kernels_run(lambda: F.solve(R))
                for kind in sweeps:
                    for direction in ("forward", "backward"):
                        assert ran(names, _sweep(kind, direction)), (kind, direction, names)
                for kind in absent:
                    assert not ran(names, _sweep(kind, "forward")) and not ran(names, _sweep(kind, "backward")), (kind, names)
            else:
                X = F.solve(R[:, :nrhs]).reshape(N, nrhs)
            check_solution(A, R[:, :nrhs], X, ref, backward=nrhs in (1, 65, 257))


# ==== device memspace =======================================================================================================
def _dev(a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")


def _kkt_solve_device(ctx, K, R, trans):
    """diffopt_b200_kkt_solve_csc with the CSC arrays, right-hand sides and solutions all in device memory."""
    capi = diffopt_b200.submodule("_capi")
    lsq = diffopt_b200.submodule("lsqr")
    colptr, rowval, nzval = lsq.julia_csc(sp.csc_matrix(K))
    N, nrhs = R.shape
    cp, rv, nz = _dev(colptr, torch.int64), _dev(rowval, torch.int64), _dev(nzval, torch.float64)
    Rd = _dev(R.T, torch.float64)                 # (nrhs, N) row-major == N x nrhs column-major
    Xd = torch.full_like(Rd, np.nan)
    torch.cuda.synchronize()
    rc = ctx.lib.diffopt_b200_kkt_solve_csc(ctx.h, N, capi.ptr(cp), capi.ptr(rv), capi.ptr(nz), int(trans), nrhs,
                                            capi.ptr(Rd), capi.ptr(Xd), capi.DEVICE)
    assert ctx.check(rc) == 0
    return Xd.cpu().numpy().T


@pytest.mark.parametrize("route", ["one_cta", "blocked", "multifrontal"])
def test_kkt_solve_csc_device_memspace(ctx, lsq, route):
    """DIFFOPT_B200_DEVICE (the Julia shim and CUDA.jl callers): the same kernels in the same order as the host call, no
    duplicate entries for the scatter's atomics to reorder -- the solution equals the host call's bit for bit."""
    K = {"one_cta": lambda: sp.csc_matrix(dense_kkt(40, 40, 20, seed=5500)),
         "blocked": lambda: sp.csc_matrix(dense_kkt(250, 250, 100, seed=5501)),
         "multifrontal": lambda: sparse_random(1100, 0.005, seed=12)}[route]()
    expect = {"one_cta": DENSE_ONE_CTA, "blocked": BL_REG32, "multifrontal": MF_ANY}[route]
    R = np.random.default_rng(13).standard_normal((K.shape[0], 70))
    for trans in (False, True):
        Xh = solve(lsq, ctx, K, R, trans)
        names, Xd = kernels_run(lambda: _kkt_solve_device(ctx, K, R, trans))
        assert ran(names, expect), names
        assert np.array_equal(Xd, Xh)
        check_solution(sp.csc_matrix(K.T) if trans else K, R, Xd, backward=False)


def test_sparse_solve_device_memspace(ctx, lsq):
    """diffopt_b200_sparse_solve with device right-hand sides and solutions: bit for bit the host call's answer."""
    capi = diffopt_b200.submodule("_capi")
    K = arrowhead(90)
    R = np.random.default_rng(14).standard_normal((K.shape[0], 129))
    F = lsq.SparseFactorization(ctx, K, trans=True)
    Xh = F.solve(R)
    Rd = _dev(R.T, torch.float64)
    Xd = torch.full_like(Rd, np.nan)
    torch.cuda.synchronize()
    ctx.check(ctx.lib.diffopt_b200_sparse_solve(ctx.h, R.shape[1], capi.ptr(Rd), capi.ptr(Xd), capi.DEVICE))
    assert np.array_equal(Xd.cpu().numpy().T, Xh)
    check_solution(sp.csc_matrix(K.T), R, Xh, backward=False)
