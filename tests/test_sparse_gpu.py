"""GPU parity tests of the multifrontal sparse direct path (diffopt_b200_sparse_setup / _sparse_solve, csrc/sparse_mf.cu)
-- `LHS \\ RHS` of QuadraticProgram.jl:486-492 for large sparse KKT systems -- against SuperLU (scipy's splu, the stand-in
for the reference's UMFPACK).  Tolerance: relative error <= 1e-8 per right-hand side (north_star, direct solves)."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import bench_data
import diffopt_b200

pytestmark = pytest.mark.gpu
RTOL_DIRECT = 1e-8


@pytest.fixture(scope="module")
def ctx():
    return diffopt_b200.Context(0)


def _check(ctx, K, nrhs, trans, seed=0, expect_method="multifrontal"):
    lsq = diffopt_b200.submodule("lsqr")
    N = K.shape[0]
    R = np.random.default_rng(seed).standard_normal((N, nrhs))
    F = lsq.SparseFactorization(ctx, K, trans=trans)
    assert F.stats["method"] == expect_method, F.stats
    X = F.solve(R)
    ref = spla.splu(sp.csc_matrix(K.T if trans else K)).solve(R)
    err = (np.linalg.norm(X - ref, axis=0) / np.linalg.norm(ref, axis=0)).max()
    assert err <= RTOL_DIRECT, (err, F.stats)
    return F


def _random_sparse(N, density, seed, weak_diag=True):
    rng = np.random.default_rng(seed)
    M = sp.random(N, N, density=density, random_state=np.random.RandomState(seed), format="csc",
                  data_rvs=lambda k: rng.standard_normal(k))
    d = rng.uniform(0.5, 2.0, N) * rng.choice([-1, 1], N) * (0.05 if weak_diag else 1.0)
    return sp.csc_matrix(M + sp.diags(d) + sp.diags(rng.uniform(1, 2, N - 1), 1) * 0.5)


@pytest.mark.parametrize("N,density,nrhs", [(1, 1.0, 1), (7, 0.5, 3), (60, 0.08, 5), (500, 0.006, 70), (3000, 0.0012, 9)])
@pytest.mark.parametrize("trans", [False, True])
def test_random_patterns(ctx, N, density, nrhs, trans):
    """General nonsymmetric patterns with a weak diagonal (pivoting inside the fronts does real work); nrhs = 70 crosses
    a 64-column tile boundary."""
    _check(ctx, _random_sparse(N, density, seed=N), nrhs, trans)


def _banded_random(N, bw, seed):
    rng = np.random.default_rng(seed)
    diags = {k: rng.standard_normal(N - abs(k)) * (rng.random(N - abs(k)) < 0.6) for k in range(-bw, bw + 1)}
    M = sp.diags([diags[k] for k in diags], list(diags), format="csc")
    # weak diagonal (partial pivoting must do real work) and a random symmetric permutation that hides the band
    M = M + sp.diags(rng.uniform(0.01, 0.1, N) * rng.choice([-1, 1], N))
    P = rng.permutation(N)
    return sp.csc_matrix(M[P][:, P])


@pytest.mark.parametrize("N,bw,nrhs", [(1, 0, 1), (50, 3, 2), (400, 17, 9), (333, 30, 3), (1000, 31, 5), (3000, 40, 33)])
def test_banded_patterns(ctx, N, bw, nrhs):
    """Permuted banded matrices with a weak diagonal (0.01 - 0.1 against entries of order 1 in the band): LHS and LHS',
    many right-hand sides, and one vector."""
    K = _banded_random(N, bw, seed=N)
    for trans in (False, True):
        F = _check(ctx, K, nrhs, trans, seed=1)
    r = np.random.default_rng(1).standard_normal((N, nrhs))[:, 0]
    assert np.allclose(F.solve(r), spla.splu(sp.csc_matrix(K.T)).solve(r), rtol=1e-7, atol=1e-10)


def test_arrow_matrix(ctx):
    """One dense row and column over a diagonal (N = 2000): no narrow band exists; the dense vertex is eliminated last.
    LHS and LHS'."""
    N = 2000
    Aw = sp.lil_matrix((N, N)); Aw.setdiag(2.0); Aw[0, :] = 1.0; Aw[:, 0] = 1.0
    for trans in (False, True):
        _check(ctx, sp.csc_matrix(Aw), 3, trans, seed=7)


def test_mpc_kkt_forward_directions(ctx):
    """BASELINE config 3 at reduced horizon (T = 300, N = 7200): the reference's LHS of an MPC QP; forward mode solves with
    LHS' (QuadraticProgram.jl:438); 16 directions against one factorisation."""
    d = bench_data.mpc_config3(T=300)
    F = _check(ctx, d["K"], 16, True, seed=2)
    assert F.stats["levels"] >= 3 and F.stats["max_front"] <= 192   # levels of GROUPED separators (3 dissection levels each)
    X = F.solve(np.eye(d["K"].shape[0])[:, :3])
    assert np.abs(d["K"].T @ X - np.eye(d["K"].shape[0])[:, :3]).max() < 1e-9


def test_portfolio_kkt_arrowhead(ctx):
    """Portfolio variant of config 3 (SURVEY 8d) at reduced size: dense budget / factor rows, 2000 assets -- an arrowhead
    no band ordering handles; dense vertices are eliminated last in one top front."""
    d = bench_data.portfolio_config3(n=2000, nfac=20, density=0.2)
    for trans in (False, True):
        _check(ctx, d["K"], 12, trans, seed=3)


def test_assembly_nodes_regroup_many_children(ctx, monkeypatch):
    """A top front with a thousand children (16 000 assets under 21 dense rows): the children are regrouped under
    assembly nodes (fronts without pivots) in two levels; same solution as with the plain one-level tree, and as SuperLU."""
    d = bench_data.portfolio_config3(n=16000, nfac=20, density=0.2)
    lsq = diffopt_b200.submodule("lsqr")
    R = np.random.default_rng(5).standard_normal((d["K"].shape[0], 70))
    F = _check(ctx, d["K"], 70, True, seed=5)
    X = F.solve(R)
    monkeypatch.setenv("DIFFOPT_B200_MF_NO_ASSEMBLY_NODES", "1")
    F0 = lsq.SparseFactorization(ctx, d["K"], trans=True)
    X0 = F0.solve(R)
    assert F.stats["levels"] == F0.stats["levels"] + 2 and F.stats["fronts"] > F0.stats["fronts"], (F.stats, F0.stats)
    assert (np.linalg.norm(X - X0, axis=0) / np.linalg.norm(X0, axis=0)).max() <= 1e-10


def test_grid_pattern_with_large_fronts(ctx):
    """2-D grid (five-point) pattern, 70 x 70: the top separators exceed what the shared-memory kernels hold, so the
    in-place global-memory path for large fronts runs too."""
    n = 70
    T = sp.diags([-1.0, 4.0, -1.0], [-1, 0, 1], shape=(n, n))
    L = sp.kron(sp.identity(n), T) + sp.kron(sp.diags([-1.0, -1.0], [-1, 1], shape=(n, n)), sp.identity(n))
    rng = np.random.default_rng(5)
    K = sp.csc_matrix(L + sp.diags(rng.standard_normal(n * n)) * 0.3)       # indefinite, nonsymmetric values below
    K = sp.csc_matrix(K + sp.triu(K, 1) * 0.25)
    F = _check(ctx, K, 10, False, seed=4)
    assert F.stats["max_front"] > 60


@pytest.mark.parametrize("diag", [0.0, 1e-5])
def test_delayed_pivots_are_merged_into_the_parent(ctx, diag):
    """Tridiagonal matrix whose pivots must come from off the diagonal (KKT-like).  diag = 0: the exactly zero diagonal is
    seen by the analysis, which pairs every such vertex with a neighbour (matching-compressed ordering) so that the pivot
    row sits in the same front.  diag = 1e-5 (weak, but above the analysis' 1e-8 test): no pairing, so a leaf whose last
    column can only be pivoted with a row of its separator fails the threshold test (|pivot| >= 1e-3 max|column|) and
    REPORTS it; the host merges such fronts into their parents and the factorisation is repeated."""
    N = 1000
    rng = np.random.default_rng(6)
    K = sp.diags([rng.uniform(1, 2, N - 1), diag * rng.uniform(1, 2, N), rng.uniform(1, 2, N - 1)], [-1, 0, 1], format="csc")
    lsq = diffopt_b200.submodule("lsqr")
    F = lsq.SparseFactorization(ctx, K)
    R = rng.standard_normal((N, 4))
    X = F.solve(R)
    ref = spla.splu(K).solve(R)
    assert (np.linalg.norm(X - ref, axis=0) / np.linalg.norm(ref, axis=0)).max() <= RTOL_DIRECT
    if diag:
        assert F.stats["method"] == "multifrontal" and F.stats["delayed_pivot_retries"] >= 1, F.stats


def test_delayed_pivots_below_assembly_nodes(ctx):
    """Arrowhead with weak diagonal entries in a few leaves (1e-5 against couplings of order 1 to the dense rows): those
    leaves fail the threshold test and report a delayed pivot; their parent is an ASSEMBLY NODE, which stands in for the top
    front -- the merge goes into the real parent and the repeated factorisation matches SuperLU."""
    n, d = 3000, 12
    rng = np.random.default_rng(8)
    diag = rng.uniform(1, 2, n) * rng.choice([-1, 1], n)
    weak = rng.choice(n, 6, replace=False)
    diag[weak] = 1e-5
    B = sp.random(n, d, density=0.3, random_state=np.random.RandomState(8), format="csc", data_rvs=lambda k: rng.uniform(0.5, 1.5, k))
    C = sp.random(d, n, density=0.3, random_state=np.random.RandomState(9), format="csc", data_rvs=lambda k: rng.uniform(0.5, 1.5, k))
    D = sp.csc_matrix(rng.standard_normal((d, d)) + 40.0 * np.eye(d))
    K = sp.bmat([[sp.diags(diag), B], [C, D]], format="csc")
    F = _check(ctx, K, 5, False, seed=8)
    assert F.stats["delayed_pivot_retries"] >= 1 and F.stats["levels"] >= 3, F.stats


def test_singular_matrix_is_reported(ctx):
    lsq = diffopt_b200.submodule("lsqr")
    S = sp.csc_matrix(np.array([[1.0, 2.0, 0.0], [1.0, 2.0, 0.0], [0.0, 1.0, 1.0]]))
    with pytest.raises(diffopt_b200.SingularException):
        lsq.SparseFactorization(ctx, S)
    Z = sp.csc_matrix(np.array([[1.0, 0.0, 0.0], [0.0, 0.0, 0.0], [0.0, 0.0, 1.0]]))
    with pytest.raises(diffopt_b200.SingularException):
        lsq.SparseFactorization(ctx, Z)


def test_solve_system_routes_large_systems_to_the_sparse_path(ctx):
    """`solve_system(::B200Solver)` binds diffopt_b200_kkt_solve_csc: beyond the dense kernel's size it must use the
    sparse factorisation instead of refusing (VERDICT r1: stale "N > 8192 ... not built yet")."""
    lsq = diffopt_b200.submodule("lsqr")
    d = bench_data.mpc_config3(T=500)          # N = 12 000
    K = d["K"]
    R = np.random.default_rng(8).standard_normal((K.shape[0], 3))
    for trans in (False, True):
        X = lsq.solve_csc(ctx, K, R, trans=trans)
        ref = spla.splu(sp.csc_matrix(K.T if trans else K)).solve(R)
        assert (np.linalg.norm(X - ref, axis=0) / np.linalg.norm(ref, axis=0)).max() <= RTOL_DIRECT
