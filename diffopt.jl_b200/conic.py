"""Host-side mirror of the reference's ConicProgram backend (src/ConicProgram/ConicProgram.jl)
on top of the C ABI.  ``ConicModel`` keeps the reference's stored quantities (x, s, y), builds the
gradient cache on the device (``_gradient_cache`` :172-255 -> ``diffopt_b200_conic_setup``) and
exposes ``forward_differentiate!`` (:257-334), ``reverse_differentiate!`` (:336-394) and the
getters (:396-443).  No arithmetic of the path runs on the CPU."""
from __future__ import annotations

import time

import numpy as np

from . import _capi
from ._capi import (CONE_DUAL_EXP, CONE_DUAL_POW, CONE_EXP, CONE_NONNEG, CONE_POW, CONE_PSD, CONE_SOC,  # noqa: F401
                    CONE_ZERO, HOST, Context, ptr)
from .lsqr import DEFAULTS, julia_csc


class ConicModel:
    """Geometric conic form  A x + s = b, s in K  with the reference's conventions:
    ``A = -coefficients`` (:179-183), ``b = constants``, ``c`` negated for MAX sense (:206-208).
    ``cone_params``: one number per cone, the exponent of each ``PowerCone`` / ``DualPowerCone`` (other entries are not
    read); None when the list has no power cone."""

    def __init__(self, ctx: Context, A, b, c, cone_types, cone_dims, cone_params=None):
        import scipy.sparse as sp
        self.ctx = ctx
        self.A = sp.csc_matrix(A, dtype=np.float64)
        self.m, self.n = self.A.shape
        self.b = np.ascontiguousarray(b, dtype=np.float64).reshape(self.m)
        self.c = np.ascontiguousarray(c, dtype=np.float64).reshape(self.n)
        self.cone_types = np.ascontiguousarray(cone_types, dtype=np.int32)
        self.cone_dims = np.ascontiguousarray(cone_dims, dtype=np.int64)
        self.cone_params = None if cone_params is None else np.ascontiguousarray(cone_params, dtype=np.float64)
        if self.cone_params is not None and self.cone_params.shape != self.cone_types.shape:
            raise ValueError("cone_params needs one entry per cone")
        self.x = np.full(self.n, np.nan)
        self.s = np.full(self.m, np.nan)
        self.y = np.full(self.m, np.nan)
        self.gradient_cache = False
        self.forw_grad_cache = None
        self.back_grad_cache = None
        self.diff_time = float("nan")
        self.tolerances = dict(DEFAULTS, maxiter=None)
        self.last_stats = None

    @classmethod
    def from_moi(cls, ctx, coefficients, constants, c, cone_types, cone_dims, max_sense=False, cone_params=None):
        """From MOI-style data (function = coefficients x + constants in K), applying the
        reference's sign handling."""
        import scipy.sparse as sp
        return cls(ctx, -sp.csc_matrix(coefficients, dtype=np.float64), constants,
                   -np.asarray(c, float) if max_sense else c, cone_types, cone_dims, cone_params)

    # MOI.set(model, VariablePrimalStart / ConstraintPrimalStart / ConstraintDualStart, ...)
    def set_variable_primal(self, x):
        self.x = np.ascontiguousarray(x, dtype=np.float64).reshape(self.n)
        self.gradient_cache = False

    def set_constraint_primal(self, s):
        self.s = np.ascontiguousarray(s, dtype=np.float64).reshape(self.m)
        self.gradient_cache = False

    def set_constraint_dual(self, y):
        self.y = np.ascontiguousarray(y, dtype=np.float64).reshape(self.m)
        self.gradient_cache = False

    def _gradient_cache(self):
        if self.gradient_cache:
            return
        if np.isnan(self.y).any():   # ConicProgram.jl:186-196
            raise ValueError("Some constraints are missing a value for the `ConstraintDualStart` attribute.")
        if np.isnan(self.s).any():
            raise ValueError("Some constraints are missing a value for the `ConstraintPrimalStart` attribute.")
        colptr, rowval, nzval = julia_csc(self.A)
        rc = self.ctx.lib.diffopt_b200_conic_setup_ex(
            self.ctx.h, self.n, self.m, ptr(colptr), ptr(rowval), ptr(nzval), ptr(self.b), ptr(self.c),
            ptr(self.x), ptr(self.s), ptr(self.y), len(self.cone_types), ptr(self.cone_types),
            ptr(self.cone_dims), ptr(self.cone_params), HOST)
        self.ctx.check(rc)
        self.setup_ms = self.ctx.last_kernel_ms
        self.gradient_cache = True

    def _tol(self):
        t = self.tolerances
        return t["atol"], t["btol"], t["conlim"], 0 if t["maxiter"] is None else int(t["maxiter"])

    def vp(self):
        self._gradient_cache()
        out = np.empty(self.m)
        self.ctx.check(self.ctx.lib.diffopt_b200_conic_get_vp(self.ctx.h, ptr(out), HOST))
        return out

    def dpi_apply(self, t, transpose=False):
        self._gradient_cache()
        t = np.ascontiguousarray(t, dtype=np.float64)
        out = np.empty(self.m)
        self.ctx.check(self.ctx.lib.diffopt_b200_conic_dpi_apply(self.ctx.h, ptr(t), int(transpose), ptr(out), HOST))
        return out

    def M_apply(self, t, transpose=False):
        self._gradient_cache()
        t = np.ascontiguousarray(t, dtype=np.float64)
        out = np.empty(self.n + self.m + 1)
        self.ctx.check(self.ctx.lib.diffopt_b200_conic_M_apply(self.ctx.h, ptr(t), int(transpose), ptr(out), HOST))
        return out

    def forward_differentiate(self, dA=None, db=None, dc=None):
        """dA: scipy sparse / dense (m x n) perturbation of the constraint *coefficients as set through
        ForwardConstraintFunction* (used un-negated, :296-305); db: constants; dc: objective."""
        import scipy.sparse as sp
        t0 = time.perf_counter()
        self._gradient_cache()
        if dA is None:
            rows = cols = vals = None
            nnz = 0
        else:
            coo = sp.coo_matrix(dA)
            rows = np.ascontiguousarray(coo.row.astype(np.int64) + 1)
            cols = np.ascontiguousarray(coo.col.astype(np.int64) + 1)
            vals = np.ascontiguousarray(coo.data, dtype=np.float64)
            nnz = vals.size
        db = None if db is None else np.ascontiguousarray(db, dtype=np.float64).reshape(self.m)
        dc = None if dc is None else np.ascontiguousarray(dc, dtype=np.float64).reshape(self.n)
        dx = np.empty(self.n)
        dz = np.empty(self.n + self.m + 1)
        stats = np.zeros(4)
        rc = self.ctx.lib.diffopt_b200_conic_forward(self.ctx.h, nnz, ptr(rows), ptr(cols), ptr(vals), ptr(db), ptr(dc),
                                                     *self._tol(), ptr(dx), ptr(dz), ptr(stats), HOST)
        self.ctx.check(rc)
        n, m = self.n, self.m
        self.forw_grad_cache = (dz[:n], dz[n:n + m], dz[n + m:], dx)
        self.last_stats = dict(istop=int(stats[0]), itn=int(stats[1]), rnorm=stats[2], arnorm=stats[3],
                               kernel_ms=self.ctx.last_kernel_ms)
        self.diff_time = time.perf_counter() - t0

    def forward_differentiate_multi(self, dAs=None, dbs=None, dcs=None, k=None):
        """k forward directions in one call (``diffopt_b200_conic_forward_multi``): dAs a list of k sparse / dense (m x n)
        matrices or None entries (zero), dbs (k, m), dcs (k, n); any may be None.  k is taken from the inputs unless
        given.  Returns dict(dx (k, n), dz (k, n+m+1), stats (k, 4)); direction j equals ``forward_differentiate`` of
        (dAs[j], dbs[j], dcs[j]) up to rounding.  The model's own caches are not touched."""
        import scipy.sparse as sp
        from .qp import coo_batch
        self._gradient_cache()
        n, m = self.n, self.m
        if k is None:
            k = next(len(v) for v in (dAs, dbs, dcs) if v is not None)
        vec = lambda v, r: None if v is None else np.ascontiguousarray(np.asarray(v, float).reshape(k, r))
        dbs, dcs = vec(dbs, m), vec(dcs, n)
        keep = None
        if dAs is not None:
            if len(dAs) != k:
                raise ValueError("dAs needs one entry per direction")
            arrs = coo_batch([sp.csr_matrix((m, n)) if M is None else M for M in dAs], k)
            keep = (arrs, _capi.CooBatch(*[a.ctypes.data for a in arrs]))
        dx = np.empty((k, n))
        dz = np.empty((k, n + m + 1))
        stats = np.zeros((k, 4))
        rc = self.ctx.lib.diffopt_b200_conic_forward_multi(self.ctx.h, k, None if keep is None else _capi.C.addressof(keep[1]),
                                                           ptr(dbs), ptr(dcs), *self._tol(), ptr(dx), ptr(dz), ptr(stats), HOST)
        self.ctx.check(rc)
        return dict(dx=dx, dz=dz, stats=stats)

    def reverse_differentiate_multi(self, dx_seeds):
        """k reverse seeds in one call (``diffopt_b200_conic_reverse_multi``): dx_seeds (k, n) -> dict(g (k, n+m+1),
        dc (k, n), db (k, m), stats (k, 4)); row j equals ``reverse_differentiate(dx_seeds[j])`` up to rounding."""
        self._gradient_cache()
        n, m = self.n, self.m
        seeds = np.ascontiguousarray(np.asarray(dx_seeds, dtype=np.float64).reshape(-1, n))
        k = seeds.shape[0]
        g = np.empty((k, n + m + 1))
        dc = np.empty((k, n))
        db = np.empty((k, m))
        stats = np.zeros((k, 4))
        rc = self.ctx.lib.diffopt_b200_conic_reverse_multi(self.ctx.h, k, ptr(seeds), *self._tol(), ptr(g), ptr(dc), ptr(db),
                                                           ptr(stats), HOST)
        self.ctx.check(rc)
        return dict(g=g, dc=dc, db=db, stats=stats)

    def reverse_differentiate(self, dx_seed):
        t0 = time.perf_counter()
        self._gradient_cache()
        seed = np.ascontiguousarray(dx_seed, dtype=np.float64).reshape(self.n)
        g = np.empty(self.n + self.m + 1)
        dc = np.empty(self.n)
        db = np.empty(self.m)
        stats = np.zeros(4)
        rc = self.ctx.lib.diffopt_b200_conic_reverse(self.ctx.h, ptr(seed), *self._tol(), ptr(g), ptr(dc), ptr(db),
                                                     ptr(stats), HOST)
        self.ctx.check(rc)
        self.back_grad_cache = dict(g=g, dc=dc, db=db)
        self.last_stats = dict(istop=int(stats[0]), itn=int(stats[1]), rnorm=stats[2], arnorm=stats[3],
                               kernel_ms=self.ctx.last_kernel_ms)
        self.diff_time = time.perf_counter() - t0

    # getters ------------------------------------------------------------------------------------
    def forward_variable_primal(self):
        return self.forw_grad_cache[3]                    # -(du - x dw), :403-412

    def reverse_objective_function(self):
        return self.back_grad_cache["dc"]                 # :396-401

    def get_db(self, rows=None):
        db = self.back_grad_cache["db"]                   # :414-428
        return db if rows is None else db[rows]

    def get_dA(self, rows):
        """g[n+I] x' - vp[I] g[1:n]'  (:430-443): an outer-product view the reference also forms lazily,
        assembled here from the device results for the requested rows only."""
        g = self.back_grad_cache["g"]
        n = self.n
        vp = self.vp()
        rows = np.atleast_1d(rows)
        return np.outer(g[n + rows], self.x) - np.outer(vp[rows], g[:n])


class ConicBatch:
    """Lock-step batch of ``ConicModel``s of equal size (``diffopt_b200_conic_batch_*``): the reference differentiates one
    problem per ``reverse_differentiate!`` call (ConicProgram.jl:336-394); a training loop makes that call once per
    sample of a minibatch.  Here every problem is analysed as usual and ONE persistent kernel advances all the LSQR
    solves -- each with its own operator, stop tests and iteration count."""

    def __init__(self, ctx: Context, models, ctas_per_problem=1):
        self.ctx = ctx
        self.models = list(models)
        self.B = len(self.models)
        self.n, self.m = self.models[0].n, self.models[0].m
        self.tolerances = dict(DEFAULTS, maxiter=None)
        ctx.check(ctx.lib.diffopt_b200_conic_batch_begin(ctx.h, self.B, int(ctas_per_problem)))
        for mdl in self.models:
            colptr, rowval, nzval = julia_csc(mdl.A)
            ctx.check(ctx.lib.diffopt_b200_conic_batch_add_ex(
                ctx.h, mdl.n, mdl.m, ptr(colptr), ptr(rowval), ptr(nzval), ptr(mdl.b), ptr(mdl.c), ptr(mdl.x), ptr(mdl.s),
                ptr(mdl.y), len(mdl.cone_types), ptr(mdl.cone_types), ptr(mdl.cone_dims), ptr(mdl.cone_params), HOST))

    def reverse_differentiate(self, dx_seeds):
        """dx_seeds: (B, n).  Returns dict(g (B, n+m+1), dc (B, n), db (B, m), stats (B, 4))."""
        B, n, m = self.B, self.n, self.m
        seeds = np.ascontiguousarray(dx_seeds, dtype=np.float64).reshape(B, n)
        g = np.empty((B, n + m + 1))
        dc = np.empty((B, n))
        db = np.empty((B, m))
        stats = np.zeros((B, 4))
        t = self.tolerances
        rc = self.ctx.lib.diffopt_b200_conic_batch_reverse(
            self.ctx.h, ptr(seeds), t["atol"], t["btol"], t["conlim"], 0 if t["maxiter"] is None else int(t["maxiter"]),
            ptr(g), ptr(dc), ptr(db), ptr(stats), HOST)
        self.ctx.check(rc)
        self.kernel_ms = self.ctx.last_kernel_ms
        return dict(g=g, dc=dc, db=db, stats=stats)
