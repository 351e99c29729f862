"""Host wrapper of ``diffopt_b200_lsqr_csc``: LSQR on an explicit sparse matrix in Julia's CSC
layout -- the ``iterative`` branch of ``solve_system`` (QuadraticProgram.jl:486-492)."""
from __future__ import annotations

import math

import numpy as np

from ._capi import HOST, Context, ptr

SQRT_EPS = math.sqrt(np.finfo(np.float64).eps)
# IterativeSolvers.lsqr defaults (see oracle/lsqr.py for the parity note)
DEFAULTS = dict(atol=SQRT_EPS, btol=SQRT_EPS, conlim=1.0 / SQRT_EPS)


def julia_csc(M):
    """scipy sparse / dense -> (colptr, rowval, nzval) 1-based int64 like SparseMatrixCSC{Float64,Int}."""
    import scipy.sparse as sp
    M = sp.csc_matrix(M, dtype=np.float64)
    M.sort_indices()
    return (M.indptr.astype(np.int64) + 1, M.indices.astype(np.int64) + 1,
            np.ascontiguousarray(M.data, dtype=np.float64))


def lsqr_csc(ctx: Context, M, rhs, trans=False, atol=None, btol=None, conlim=None, maxiter=None):
    """x = argmin ||M x - rhs|| (or M' when ``trans``) from x0 = 0.  Returns (x, stats)."""
    nrows, ncols = M.shape
    colptr, rowval, nzval = julia_csc(M)
    rhs = np.ascontiguousarray(rhs, dtype=np.float64)
    x = np.empty(nrows if trans else ncols)
    stats = np.zeros(4)
    rc = ctx.lib.diffopt_b200_lsqr_csc(
        ctx.h, nrows, ncols, ptr(colptr), ptr(rowval), ptr(nzval), int(trans), ptr(rhs),
        DEFAULTS["atol"] if atol is None else atol, DEFAULTS["btol"] if btol is None else btol,
        DEFAULTS["conlim"] if conlim is None else conlim, 0 if maxiter is None else int(maxiter),
        ptr(x), ptr(stats), HOST)
    ctx.check(rc)
    return x, dict(istop=int(stats[0]), itn=int(stats[1]), rnorm=stats[2], arnorm=stats[3])


def solve_csc(ctx: Context, M, rhs, trans=False):
    """Direct branch of ``solve_system`` (``LHS \\ RHS``, QuadraticProgram.jl:490) through
    ``diffopt_b200_kkt_solve_csc``: one pivoted LU on the device, ``rhs`` may hold many columns
    (N x nrhs).  Raises ``SingularException`` on an exactly zero pivot like the reference."""
    from ._capi import SingularException
    N = M.shape[0]
    colptr, rowval, nzval = julia_csc(M)
    rhs = np.asarray(rhs, dtype=np.float64)
    one = rhs.ndim == 1
    R = np.asfortranarray(rhs.reshape(N, -1))
    X = np.empty_like(R, order="F")
    rc = ctx.lib.diffopt_b200_kkt_solve_csc(ctx.h, N, ptr(colptr), ptr(rowval), ptr(nzval), int(trans), R.shape[1],
                                            ptr(R), ptr(X), HOST)
    ctx.check(rc)
    if rc > 0:
        raise SingularException(rc)
    return X[:, 0].copy() if one else X


def sparse_analyze(M, trans=False):
    """Host-only ordering + symbolic factorisation of a pattern (``diffopt_b200_sparse_analyze``; no GPU needed)."""
    from ._capi import load
    colptr, rowval, nzval = julia_csc(M)
    st = np.zeros(8)
    rc = load().diffopt_b200_sparse_analyze(M.shape[0], ptr(colptr), ptr(rowval), ptr(nzval), int(trans), ptr(st))
    if rc != 0:
        raise RuntimeError(f"sparse_analyze failed ({rc})")
    return dict(fronts=int(st[1]), levels=int(st[2]), max_front=int(st[3]), nnz_lu=int(st[4]), factor_flops=float(st[5]),
                analysis_ms=float(st[6]), launches=int(st[7]))


class SparseFactorization:
    """``diffopt_b200_sparse_setup`` / ``_sparse_solve``: one factorisation of a large sparse KKT matrix (or of its
    adjoint) on the device (multifrontal LU), reused for any number of right-hand sides -- the
    direct ``LHS \\ RHS`` of QuadraticProgram.jl:490 for systems beyond the dense kernels (BASELINE config 3)."""

    def __init__(self, ctx: Context, M, trans=False):
        from ._capi import SingularException
        self.ctx = ctx
        self.N = M.shape[0]
        colptr, rowval, nzval = julia_csc(M)
        rc = ctx.lib.diffopt_b200_sparse_setup(ctx.h, self.N, ptr(colptr), ptr(rowval), ptr(nzval), int(trans), None)
        ctx.check(rc)
        if rc > 0:
            raise SingularException(rc)
        self.factor_ms = ctx.last_kernel_ms
        st = np.zeros(8)
        ctx.check(ctx.lib.diffopt_b200_sparse_stats(ctx.h, ptr(st)))
        self.stats = dict(method={0: "none", 2: "multifrontal"}[int(st[0])], fronts=int(st[1]), levels=int(st[2]),
                          max_front=int(st[3]), nnz_lu=int(st[4]), factor_flops=float(st[5]), analysis_ms=float(st[6]),
                          delayed_pivot_retries=int(st[7]))

    def solve(self, rhs):
        rhs = np.asarray(rhs, dtype=np.float64)
        one = rhs.ndim == 1
        R = np.asfortranarray(rhs.reshape(self.N, -1))
        X = np.empty_like(R, order="F")
        self.ctx.check(self.ctx.lib.diffopt_b200_sparse_solve(self.ctx.h, R.shape[1], ptr(R), ptr(X), HOST))
        self.solve_ms = self.ctx.last_kernel_ms
        return X[:, 0].copy() if one else X
