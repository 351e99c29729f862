"""Host-side mirror of the reference's QuadraticProgram backend on top of the C ABI.

``QPModel`` follows ``DiffOpt.QuadraticProgram.Model`` (src/QuadraticProgram/QuadraticProgram.jl):
same stored quantities (``x``, ``λ``, ``ν`` with the reference's sign flip, :156-180), the same
``forward_differentiate!`` / ``reverse_differentiate!`` entry points, the same getters
(ForwardVariablePrimal :299-305, ReverseObjectiveFunction :448-458, _get_dA/_get_db :307-314,
:461-473) and the same error behaviour (SingularException from the direct solve).  All
arithmetic happens in the CUDA library; nothing here computes a solve on the CPU.

``QPBatch`` is the batched form (B independent instances) the GPU path is built for.
"""
from __future__ import annotations

import time

import numpy as np

from . import _capi
from ._capi import DEVICE, HOST, Context, SingularException, ptr


def colmajor(X, rows, cols, B=None):
    """(B, rows, cols) or (rows, cols) logical matrices -> instance-major, column-major buffer."""
    X = np.asarray(X, dtype=np.float64)
    if B is None:
        X = X.reshape(1, rows, cols)
    else:
        X = X.reshape(B, rows, cols)
    return np.ascontiguousarray(X.transpose(0, 2, 1))


def from_colmajor(buf, rows, cols):
    return np.asarray(buf).reshape(-1, cols, rows).transpose(0, 2, 1)


class QPBatch:
    """B independent QPs  min ½z'Qz+q'z  s.t. Gz<=h, Az=b, already solved: (z, lam, nu).

    Arrays are logical (B, rows, cols) / (B, len) numpy arrays; ``lam``/``nu`` follow the
    reference's convention (negated MOI duals).  ``solve`` = one fused launch doing KKT assembly,
    one LU factorisation, the forward solve with LHS' and the reverse solve with LHS.
    """

    def __init__(self, ctx: Context, Q, G, A, h, z, lam, nu):
        self.ctx = ctx
        z = np.ascontiguousarray(z, dtype=np.float64)
        self.B, self.n = z.shape
        self.m = 0 if lam is None else np.asarray(lam).reshape(self.B, -1).shape[1]
        self.p = 0 if nu is None else np.asarray(nu).reshape(self.B, -1).shape[1]
        B, n, m, p = self.B, self.n, self.m, self.p
        self.N = n + m + p
        self.z = z
        self.lam = np.ascontiguousarray(np.asarray(lam, float).reshape(B, m)) if m else np.zeros((B, 0))
        self.nu = np.ascontiguousarray(np.asarray(nu, float).reshape(B, p)) if p else np.zeros((B, 0))
        self.h = np.ascontiguousarray(np.asarray(h, float).reshape(B, m)) if m else np.zeros((B, 0))
        self.Qc = colmajor(Q, n, n, B)
        self.Gc = colmajor(G, m, n, B) if m else None
        self.Ac = colmajor(A, p, n, B) if p else None
        rc = ctx.lib.diffopt_b200_qp_batch_setup(
            ctx.h, B, n, m, p, ptr(self.Qc), ptr(self.Gc), ptr(self.Ac), ptr(self.h) if m else None,
            ptr(self.z), ptr(self.lam) if m else None, ptr(self.nu) if p else None, HOST)
        ctx.check(rc)
        self.info = np.zeros(B, dtype=np.int32)

    def _raise_if_singular(self, rc):
        self.ctx.check(rc)
        if rc > 0:
            b = rc - 1
            raise SingularException(int(self.info[b]), instance=b)

    def reverse(self, dl_dz):
        seed = np.ascontiguousarray(np.asarray(dl_dz, float).reshape(self.B, self.n))
        out = np.empty((self.B, self.N))
        rc = self.ctx.lib.diffopt_b200_qp_batch_reverse(self.ctx.h, ptr(seed), ptr(out), ptr(self.info), HOST)
        self._raise_if_singular(rc)
        return self._split(out)

    def forward(self, dQ=None, dq=None, dG=None, dh=None, dA=None, db=None):
        B, n, m, p = self.B, self.n, self.m, self.p
        cm = lambda X, r: None if X is None or r == 0 else colmajor(X, r, n, B)
        vec = lambda v, k: None if v is None or k == 0 else np.ascontiguousarray(np.asarray(v, float).reshape(B, k))
        bufs = [cm(dQ, n), vec(dq, n), cm(dG, m), vec(dh, m), cm(dA, p), vec(db, p)]
        out = np.empty((B, self.N))
        rc = self.ctx.lib.diffopt_b200_qp_batch_forward(self.ctx.h, *[ptr(x) for x in bufs], ptr(out),
                                                        ptr(self.info), HOST)
        self._raise_if_singular(rc)
        return self._split(out)

    def factorize(self):
        """``diffopt_b200_qp_batch_factorize``: keep every instance's LDL' factor on the device for ``reverse_multi`` /
        ``forward_multi`` (until the next setup).  Raises SingularException for a singular instance (``info`` is kept: the
        multi calls raise for the same instance)."""
        rc = self.ctx.lib.diffopt_b200_qp_batch_factorize(self.ctx.h, ptr(self.info), HOST)
        self._raise_if_singular(rc)

    def reverse_multi(self, seeds):
        """k reverse seeds per instance, ``seeds`` (B, k, n) -> (dz, dλ, dν), each (B, k, ·): one ``reverse`` per seed."""
        seeds = np.asarray(seeds, float)
        k = seeds.shape[1]
        seeds = np.ascontiguousarray(seeds.reshape(self.B, k, self.n))
        out = np.empty((self.B, k, self.N))
        rc = self.ctx.lib.diffopt_b200_qp_batch_reverse_multi(self.ctx.h, k, ptr(seeds), ptr(out), HOST)
        self._raise_if_singular(rc)
        return self._split_multi(out)

    def forward_multi(self, k, dQ=None, dq=None, dG=None, dh=None, dA=None, db=None):
        """k forward directions per instance: dq (B, k, n), dh (B, k, m), db (B, k, p); dQ, dG, dA as B*k scipy.sparse
        matrices in slot order (direction j of instance b at b*k + j, see ``coo_batch``); any may be None (zero).
        Returns (dz, dλ, dν), each (B, k, ·): one ``forward`` per direction."""
        B, n, m, p = self.B, self.n, self.m, self.p
        vec = lambda v, r: None if v is None or r == 0 else np.ascontiguousarray(np.asarray(v, float).reshape(B, k, r))
        keep = []

        def coo(mats, rows):
            arrs = coo_batch(mats, B * k) if rows else None
            if arrs is None:
                return None
            st = _capi.CooBatch(*[a.ctypes.data for a in arrs])
            keep.append((arrs, st))
            return _capi.C.addressof(st)
        dvecs = [vec(dq, n), vec(dh, m), vec(db, p)]
        out = np.empty((B, k, self.N))
        rc = self.ctx.lib.diffopt_b200_qp_batch_forward_multi(self.ctx.h, k, coo(dQ, n), ptr(dvecs[0]), coo(dG, m), ptr(dvecs[1]),
                                                              coo(dA, p), ptr(dvecs[2]), ptr(out), HOST)
        self._raise_if_singular(rc)
        return self._split_multi(out)

    def _split_multi(self, out):
        n, m = self.n, self.m
        return out[..., :n], out[..., n:n + m], out[..., n + m:]

    def param_grads(self, rev, reduce_over_batch=False):
        """dQ, dq, dG, dh, dA, db from rev = concatenated (dz, dlam, dnu) (B, N)."""
        B, n, m, p = self.B, self.n, self.m, self.p
        rev = np.ascontiguousarray(np.asarray(rev, float).reshape(B, self.N))
        k = 1 if reduce_over_batch else B
        outs = [np.empty((k, n, n)), np.empty((k, n)), np.empty((k, n, m)), np.empty((k, m)),
                np.empty((k, n, p)), np.empty((k, p))]
        rc = self.ctx.lib.diffopt_b200_qp_batch_param_grads(self.ctx.h, ptr(rev), int(reduce_over_batch),
                                                            *[ptr(o) for o in outs], HOST)
        self.ctx.check(rc)
        dQ, dq, dG, dh, dA, db = outs
        res = (dQ.transpose(0, 2, 1), dq, dG.transpose(0, 2, 1), dh, dA.transpose(0, 2, 1), db)
        return tuple(r[0] for r in res) if reduce_over_batch else res

    def _split(self, out):
        n, m = self.n, self.m
        return out[:, :n], out[:, n:n + m], out[:, n + m:]


def solve_batch(ctx, Q, G, A, h, z, lam, nu, fwd_dir=None, seed=None):
    """Fused one-shot call (``diffopt_b200_qp_batch_solve``).  ``fwd_dir`` = (dQ,dq,dG,dh,dA,db)."""
    z = np.ascontiguousarray(z, dtype=np.float64)
    B, n = z.shape
    m = 0 if lam is None else np.asarray(lam).reshape(B, -1).shape[1]
    p = 0 if nu is None else np.asarray(nu).reshape(B, -1).shape[1]
    N = n + m + p
    cm = lambda X, r: None if X is None or r == 0 else colmajor(X, r, n, B)
    vec = lambda v, k: None if v is None or k == 0 else np.ascontiguousarray(np.asarray(v, float).reshape(B, k))
    args = [cm(Q, n), cm(G, m), cm(A, p), vec(h, m), z, vec(lam, m), vec(nu, p)]
    if fwd_dir is not None:
        dQ, dq, dG, dh, dA, db = fwd_dir
        args += [cm(dQ, n), vec(dq, n), cm(dG, m), vec(dh, m), cm(dA, p), vec(db, p)]
        fwd = np.empty((B, N))
    else:
        args += [None] * 6
        fwd = None
    rev = None
    sd = None
    if seed is not None:
        sd = vec(seed, n)
        rev = np.empty((B, N))
    info = np.zeros(B, dtype=np.int32)
    rc = ctx.lib.diffopt_b200_qp_batch_solve(ctx.h, B, n, m, p, *[ptr(a) for a in args], ptr(sd), ptr(fwd),
                                             ptr(rev), ptr(info), HOST)
    ctx.check(rc)
    return fwd, rev, info


def coo_batch(mats, B, shared=False):
    """Per-instance sparse matrices (a list of B scipy.sparse matrices, or ONE matrix with ``shared``) -> the arrays of a
    ``diffopt_b200_coo_batch``: 0-based offsets, 1-based (I, J) triplets, values -- what the reference's ``_fill`` collects
    (src/diff_opt.jl:594-656).  ``None`` -> None (a zero matrix)."""
    if mats is None:
        return None
    import scipy.sparse as sp
    mats = [mats] if shared else list(mats)
    assert len(mats) == (1 if shared else B)
    coos = [sp.coo_matrix(M) for M in mats]
    ptr = np.zeros(len(coos) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([c.nnz for c in coos])
    cat = lambda xs, dt: np.ascontiguousarray(np.concatenate(xs).astype(dt)) if xs else np.zeros(0, dt)
    return (ptr, cat([c.row + 1 for c in coos], np.int64), cat([c.col + 1 for c in coos], np.int64),
            cat([c.data for c in coos], np.float64))


def solve_batch_coo(ctx, Q, G, A, h, z, lam, nu, dQ=None, dq=None, dG=None, dh=None, dA=None, db=None, seed=None,
                    shared_direction=False):
    """``diffopt_b200_qp_batch_solve_coo``: forward (and optionally reverse) sensitivities with the direction matrices given
    as sparse triplets (lists of scipy.sparse matrices, one per instance; see ``coo_batch``)."""
    z = np.ascontiguousarray(z, dtype=np.float64)
    B, n = z.shape
    m = 0 if lam is None else np.asarray(lam).reshape(B, -1).shape[1]
    p = 0 if nu is None else np.asarray(nu).reshape(B, -1).shape[1]
    N = n + m + p
    cm = lambda X, r: None if X is None or r == 0 else colmajor(X, r, n, B)
    vec = lambda v, k: None if v is None or k == 0 else np.ascontiguousarray(np.asarray(v, float).reshape(B, k))
    args = [cm(Q, n), cm(G, m), cm(A, p), vec(h, m), z, vec(lam, m), vec(nu, p)]
    keep = []

    def coo(mats, rows):
        arrs = coo_batch(mats, B, shared_direction) if rows else None
        if arrs is None:
            return None
        keep.append(arrs)
        st = _capi.CooBatch(*[a.ctypes.data for a in arrs])
        keep.append(st)
        return _capi.C.addressof(st)
    dvecs = [vec(dq, n), vec(dh, m), vec(db, p)]
    sd = vec(seed, n) if seed is not None else None
    fwd = np.empty((B, N))
    rev = np.empty((B, N)) if seed is not None else None
    info = np.zeros(B, dtype=np.int32)
    rc = ctx.lib.diffopt_b200_qp_batch_solve_coo(
        ctx.h, B, n, m, p, *[ptr(a) for a in args], coo(dQ, n), ptr(dvecs[0]), coo(dG, m), ptr(dvecs[1]), coo(dA, p),
        ptr(dvecs[2]), ptr(sd), ptr(fwd), ptr(rev), ptr(info), HOST, _capi.QP_SHARED_DIRECTION if shared_direction else 0)
    ctx.check(rc)
    return fwd, rev, info


def pack_lower(X):
    """(B, n, n) symmetric matrices -> (B, n(n+1)/2) packed lower triangles, column by column (DIFFOPT_QP_PACKED_Q)."""
    X = np.asarray(X, dtype=np.float64)
    n = X.shape[-1]
    r, c = np.tril_indices(n)
    order = np.lexsort((r, c))           # column-major order of the lower triangle
    return np.ascontiguousarray(X.reshape(-1, n, n)[:, r[order], c[order]])


def solve_batch_ex(ctx, Q, G, A, h, z, lam, nu, fwd_dir=None, seed=None, shared_matrices=False, shared_direction=False,
                   packed_q=False):
    """``diffopt_b200_qp_batch_solve_ex``: like ``solve_batch`` with batch-invariant Q, G, A (``shared_matrices``: pass ONE
    instance, shape (n, n) / (m, n) / (p, n)), a batch-invariant forward direction dQ, dG, dA (``shared_direction``) and
    Q / dQ sent as packed lower triangles (``packed_q``)."""
    z = np.ascontiguousarray(z, dtype=np.float64)
    B, n = z.shape
    m = 0 if lam is None else np.asarray(lam).reshape(B, -1).shape[1]
    p = 0 if nu is None else np.asarray(nu).reshape(B, -1).shape[1]
    N = n + m + p
    def mat(X, r, shared, sym=False):
        if X is None or r == 0:
            return None
        k = 1 if shared else B
        if sym and packed_q:
            return pack_lower(np.asarray(X, float).reshape(k, n, n))
        return colmajor(np.asarray(X, float).reshape(k, r, n), r, n, k)
    vec = lambda v, k: None if v is None or k == 0 else np.ascontiguousarray(np.asarray(v, float).reshape(B, k))
    args = [mat(Q, n, shared_matrices, True), mat(G, m, shared_matrices), mat(A, p, shared_matrices), vec(h, m), z,
            vec(lam, m), vec(nu, p)]
    fwd = rev = sd = None
    if fwd_dir is not None:
        dQ, dq, dG, dh, dA, db = fwd_dir
        args += [mat(dQ, n, shared_direction, True), vec(dq, n), mat(dG, m, shared_direction), vec(dh, m),
                 mat(dA, p, shared_direction), vec(db, p)]
        fwd = np.empty((B, N))
    else:
        args += [None] * 6
    if seed is not None:
        sd = vec(seed, n)
        rev = np.empty((B, N))
    info = np.zeros(B, dtype=np.int32)
    flags = (_capi.QP_SHARED_MATRICES if shared_matrices else 0) | (_capi.QP_SHARED_DIRECTION if shared_direction else 0) | \
        (_capi.QP_PACKED_Q if packed_q else 0)
    rc = ctx.lib.diffopt_b200_qp_batch_solve_ex(ctx.h, B, n, m, p, *[ptr(a) for a in args], ptr(sd), ptr(fwd), ptr(rev),
                                                ptr(info), HOST, flags)
    ctx.check(rc)
    return fwd, rev, info


def solve_batch_lsqr(ctx, G, A, h, z, lam, nu, fwd_dir=None, seed=None, shared_matrices=False, atol=None, btol=None,
                     conlim=None, maxiter=None):
    """``diffopt_b200_qp_batch_solve_lsqr``: the reference's LSQR branch (Q = 0, every LP) for a batch, one CTA per
    instance.  Arguments as ``solve_batch_ex`` without Q; ``fwd_dir = (dQ, dq, dG, dh, dA, db)`` (any entry may be None).
    Tolerances default to ``lsqr.DEFAULTS`` (IterativeSolvers' values), ``maxiter`` to n + m + p.  Returns
    ``(fwd (B, N) or None, rev (B, N) or None, stats (B, 2, 4))``, stats = (istop, itn, rnorm, arnorm) of the forward,
    then the reverse solve.  Singular KKT matrices give LSQR's minimum-norm answer, as in the reference."""
    from .lsqr import DEFAULTS
    z = np.ascontiguousarray(z, dtype=np.float64)
    B, n = z.shape
    m = 0 if lam is None else np.asarray(lam).reshape(B, -1).shape[1]
    p = 0 if nu is None else np.asarray(nu).reshape(B, -1).shape[1]
    N = n + m + p
    def mat(X, r, k):
        return None if X is None or r == 0 else colmajor(np.asarray(X, float).reshape(k, r, n), r, n, k)
    vec = lambda v, k: None if v is None or k == 0 else np.ascontiguousarray(np.asarray(v, float).reshape(B, k))
    km = 1 if shared_matrices else B
    args = [mat(G, m, km), mat(A, p, km), vec(h, m), z, vec(lam, m), vec(nu, p)]
    fwd = rev = sd = None
    if fwd_dir is not None:
        dQ, dq, dG, dh, dA, db = fwd_dir
        args += [mat(dQ, n, B), vec(dq, n), mat(dG, m, B), vec(dh, m), mat(dA, p, B), vec(db, p)]
        fwd = np.empty((B, N))
    else:
        args += [None] * 6
    if seed is not None:
        sd = vec(seed, n)
        rev = np.empty((B, N))
    stats = np.zeros((B, 2, 4))
    rc = ctx.lib.diffopt_b200_qp_batch_solve_lsqr(
        ctx.h, B, n, m, p, *[ptr(a) for a in args], ptr(sd),
        DEFAULTS["atol"] if atol is None else atol, DEFAULTS["btol"] if btol is None else btol,
        DEFAULTS["conlim"] if conlim is None else conlim, 0 if maxiter is None else int(maxiter),
        ptr(fwd), ptr(rev), ptr(stats), HOST, _capi.QP_SHARED_MATRICES if shared_matrices else 0)
    ctx.check(rc)
    return fwd, rev, stats


def shared_param_grads(ctx, z, lam, nu, rev, allreduce=False, flat=False):
    """``diffopt_b200_qp_batch_shared_grads``: batch sums of the reverse-mode parameter gradients (dQ, dq, dG, dh, dA, db)
    for parameters shared by all instances; ``allreduce`` adds the NCCL all-reduce over the ranks of
    ``sharding.nccl_init``.  Returns logical (row-major) arrays like ``QPBatch.param_grads(reduce_over_batch=True)``."""
    z = np.ascontiguousarray(z, dtype=np.float64)
    B, n = z.shape
    m = 0 if lam is None else np.asarray(lam).reshape(B, -1).shape[1]
    p = 0 if nu is None else np.asarray(nu).reshape(B, -1).shape[1]
    vec = lambda v, k: None if v is None or k == 0 else np.ascontiguousarray(np.asarray(v, float).reshape(B, k))
    rev = np.ascontiguousarray(np.asarray(rev, float).reshape(B, n + m + p))
    per = n * n + n + m * n + m + p * n + p
    out = np.empty(per)
    rc = ctx.lib.diffopt_b200_qp_batch_shared_grads(ctx.h, B, n, m, p, ptr(z), ptr(vec(lam, m)), ptr(vec(nu, p)), ptr(rev),
                                                    ptr(out), HOST, _capi.QP_ALLREDUCE if allreduce else 0)
    ctx.check(rc)
    return out if flat else unflatten_param_grads(out, n, m, p)


def flat_index(n, m, p, block, i=0, j=0):
    """1-based position of a gradient entry inside the flat block [dQ | dq | dG | dh | dA | db] (matrices column-major):
    ``block`` in "dQ" (i, j), "dq" (i), "dG" (row i, variable j), "dh" (i), "dA" (row i, variable j), "db" (i); i, j 0-based."""
    off = {"dQ": 0, "dq": n * n, "dG": n * n + n, "dh": n * n + n + m * n, "dA": n * n + n + m * n + m,
           "db": n * n + n + m * n + m + p * n}[block]
    rows = {"dQ": n, "dG": m, "dA": p}.get(block)
    return off + (i + j * rows if rows is not None else i) + 1


def parameter_pullback(ctx, terms, flat, nparams):
    """``diffopt_b200_param_pullback``: reverse-mode accumulation into parameters (src/parameters.jl:341-534).  ``terms``:
    iterable of (parameter (0-based), flat index (1-based, ``flat_index``), coefficient); ``flat``: the gradient block of
    ``shared_param_grads(..., flat=True)`` (numpy array, or a device tensor consumed in place)."""
    terms = list(terms)
    tp = np.ascontiguousarray([t[0] + 1 for t in terms], dtype=np.int64)
    ti = np.ascontiguousarray([t[1] for t in terms], dtype=np.int64)
    tc = np.ascontiguousarray([t[2] for t in terms], dtype=np.float64)
    out = np.empty(nparams)
    on_device = hasattr(flat, "data_ptr")
    nflat = int(flat.numel()) if on_device else int(np.asarray(flat).size)
    if not on_device:
        flat = np.ascontiguousarray(flat, dtype=np.float64)
    if on_device:
        import torch
        dout = torch.empty(nparams, dtype=torch.float64, device=flat.device)
        rc = ctx.lib.diffopt_b200_param_pullback(ctx.h, len(terms), ptr(tp), ptr(ti), ptr(tc), nflat, ptr(flat), nparams, ptr(dout), 1)
        ctx.check(rc)
        return dout
    rc = ctx.lib.diffopt_b200_param_pullback(ctx.h, len(terms), ptr(tp), ptr(ti), ptr(tc), nflat, ptr(flat), nparams, ptr(out), HOST)
    ctx.check(rc)
    return out


def unflatten_param_grads(flat, n, m, p):
    """[dQ | dq | dG | dh | dA | db] (matrices column-major) -> logical arrays."""
    o = 0
    def take(k):
        nonlocal o
        v = flat[o:o + k]
        o += k
        return v
    dQ = take(n * n).reshape(n, n).T
    dq = take(n)
    dG = take(m * n).reshape(n, m).T
    dh = take(m)
    dA = take(p * n).reshape(n, p).T
    db = take(p)
    return dQ, dq, dG, dh, dA, db


class QPModel:
    """Single-problem backend with the reference's ``AbstractModel`` surface (array level).

    ``linear_solver`` plays the role of the ``LinearAlgebraSolver`` attribute
    (QuadraticProgram.jl:476-502): ``None`` = default rule (LSQR iff norm(Q) == 0, else direct).
    """

    def __init__(self, ctx: Context, Q, q, G, h, A, b):
        self.ctx = ctx
        self.Q = np.atleast_2d(np.asarray(Q, float))
        self.n = self.Q.shape[0]
        self.q = np.asarray(q, float).reshape(self.n)
        self.G = np.asarray(G, float).reshape(-1, self.n)
        self.h = np.asarray(h, float).reshape(-1)
        self.A = np.asarray(A, float).reshape(-1, self.n)
        self.b = np.asarray(b, float).reshape(-1)
        self.m, self.p = self.G.shape[0], self.A.shape[0]
        self.x = np.full(self.n, np.nan)
        self.lam = np.full(self.m, np.nan)   # λ = -ConstraintDual(<=)
        self.nu = np.full(self.p, np.nan)    # ν = -ConstraintDual(==)
        self.forw_grad_cache = None
        self.back_grad_cache = None
        self.diff_time = float("nan")
        self.iterative_tolerances = dict(atol=None, btol=None, conlim=None, maxiter=None)

    # -- MOI.set(model, VariablePrimalStart / ConstraintDualStart, ...) -------------------------
    def set_variable_primal(self, x):
        self.x = np.asarray(x, float).reshape(self.n).copy()

    def set_constraint_dual_le(self, moi_dual):
        self.lam = -np.asarray(moi_dual, float).reshape(self.m)     # QuadraticProgram.jl:173-180

    def set_constraint_dual_eq(self, moi_dual):
        self.nu = -np.asarray(moi_dual, float).reshape(self.p)      # QuadraticProgram.jl:164-171

    # -- the two differentiation entry points -----------------------------------------------------
    BATCHED_ORDER_MAX = 200   # n + p above which a single instance no longer fits the batched fast path

    def _iterative(self):
        return float(np.linalg.norm(self.Q)) == 0.0                 # `norm(Q) ≈ 0`, :333/:436

    def _lhs_csc(self):
        """create_LHS_matrix in Julia's CSC layout (1-based), built on the host like the reference
        (packing is host work, SURVEY.md §2); only the LSQR branch needs it explicitly."""
        import scipy.sparse as sp
        n, m, p = self.n, self.m, self.p
        Q, G, A = sp.csc_matrix(self.Q), sp.csc_matrix(self.G), sp.csc_matrix(self.A)
        D = sp.diags(self.G @ self.x - self.h) if m else sp.csc_matrix((0, 0))
        K = sp.bmat([[Q, G.T @ sp.diags(self.lam) if m else None, A.T if p else None],
                     [G if m else None, D if m else None, None],
                     [A if p else None, None, sp.csc_matrix((p, p)) if p else None]], format="csc")
        K.sort_indices()
        return K

    def _solve(self, fwd_dir=None, seed=None):
        from .lsqr import lsqr_csc
        if any(np.isnan(v).any() for v in (self.x, self.lam, self.nu)):
            raise ValueError("primal/dual start values are missing")
        if self._iterative():
            K = self._lhs_csc()
            N = K.shape[0]
            tol = {k: v for k, v in self.iterative_tolerances.items() if v is not None}
            if seed is not None:
                rhs = np.zeros(N)
                rhs[:self.n] = seed
                return -lsqr_csc(self.ctx, K, rhs, trans=False, **tol)[0]
            rhs = self._forward_rhs(*fwd_dir)
            return -lsqr_csc(self.ctx, K, rhs, trans=True, **tol)[0]
        if self.n + self.p > self.BATCHED_ORDER_MAX:
            # ONE large dense QP: the batched kernels keep an instance in one CTA's shared memory (reduced order <= ~216);
            # beyond that the reference's own route -- LHS assembled on the host, `LHS \ RHS` (QuadraticProgram.jl:335, :438)
            # -- goes through the solve_system drop-in, i.e. the blocked LU over the whole GPU (kkt_dense.cu)
            from .lsqr import solve_csc
            K = self._lhs_csc()
            if seed is not None:
                rhs = np.zeros(K.shape[0])
                rhs[:self.n] = seed
                return -solve_csc(self.ctx, K, rhs, trans=False)
            return -solve_csc(self.ctx, K, self._forward_rhs(*fwd_dir), trans=True)
        one = lambda v: None if v is None else np.asarray(v, float)[None]
        fd = None if fwd_dir is None else tuple(one(v) for v in fwd_dir)
        fwd, rev, info = solve_batch(self.ctx, self.Q[None], self.G[None] if self.m else None,
                                     self.A[None] if self.p else None, self.h[None], self.x[None],
                                     self.lam[None], self.nu[None], fwd_dir=fd,
                                     seed=None if seed is None else np.asarray(seed, float)[None])
        if info[0] != 0:
            raise SingularException(int(info[0]))
        return (fwd if seed is None else rev)[0]

    def _forward_rhs(self, dQ, dq, dG, dh, dA, db):
        # only used to hand the LSQR branch its right-hand side (:429-433); tiny host matvecs,
        # the same packing step the reference does in Julia before calling solve_system
        z, lam, nu = self.x, self.lam, self.nu
        return np.concatenate([dQ @ z + dq + dG.T @ lam + dA.T @ nu, lam * (dG @ z) - lam * dh, dA @ z - db])

    def reverse_differentiate(self, dl_dz):
        t0 = time.perf_counter()
        x = self._solve(seed=np.asarray(dl_dz, float).reshape(self.n))
        n, m = self.n, self.m
        self.back_grad_cache = (x[:n], x[n:n + m], x[n + m:])
        self.diff_time = time.perf_counter() - t0

    def forward_differentiate(self, dQ=None, dq=None, dG=None, dh=None, dA=None, db=None):
        t0 = time.perf_counter()
        n, m, p = self.n, self.m, self.p
        z = lambda v, shape: np.zeros(shape) if v is None else np.asarray(v, float).reshape(shape)
        sparse = any(hasattr(M, "tocoo") for M in (dQ, dG, dA))
        if sparse and not self._iterative():
            # the reference's own packing: sparse(I, J, V) per matrix (QuadraticProgram.jl:396-424) -> triplets to the device
            fwd, _, info = solve_batch_coo(self.ctx, self.Q[None], self.G[None] if m else None, self.A[None] if p else None,
                                           self.h[None], self.x[None], self.lam[None], self.nu[None],
                                           dQ=None if dQ is None else [dQ], dq=z(dq, n)[None], dG=None if dG is None else [dG],
                                           dh=z(dh, m)[None], dA=None if dA is None else [dA], db=z(db, p)[None])
            if info[0] != 0:
                raise SingularException(int(info[0]))
            x = fwd[0]
        else:
            dense = lambda M: M.toarray() if hasattr(M, "toarray") else M
            d = (z(dense(dQ), (n, n)), z(dq, n), z(dense(dG), (m, n)), z(dh, m), z(dense(dA), (p, n)), z(db, p))
            x = self._solve(fwd_dir=d)
        self.forw_grad_cache = (x[:n], x[n:n + m], x[n + m:])
        self.diff_time = time.perf_counter() - t0

    # -- getters ------------------------------------------------------------------------------------
    def forward_variable_primal(self):
        return self.forw_grad_cache[0]

    def reverse_objective_function(self):
        """(dq, dQ) = (∇z, (∇z z' + z ∇z')/2)   QuadraticProgram.jl:448-458."""
        dz = self.back_grad_cache[0]
        return dz, 0.5 * (np.outer(dz, self.x) + np.outer(self.x, dz))

    def get_db_le(self, i):
        return self.lam[i] * self.back_grad_cache[1][i]            # :307-311

    def get_db_eq(self, i):
        return self.back_grad_cache[2][i]                          # :312-314

    def get_dA_eq(self, i):
        dz, _, dnu = self.back_grad_cache
        return dnu[i] * self.x + self.nu[i] * dz                   # :461-466

    def get_dA_le(self, i):
        dz, dlam, _ = self.back_grad_cache
        l = self.lam[i]
        return l * dlam[i] * self.x + l * dz                       # :467-473


def poi_terms(n, m, p, constraints, objective=None, param_values=None):
    """Term triplets for ``parameter_pullback`` from parametric functions as ParametricOptInterface holds them
    (src/parameters.jl:341-534).  ``constraints``: list of dicts with ``row`` = ("ineq", i) or ("eq", i) (row of G / A the
    inner constraint became, already in LessThan / EqualTo form) and the term lists ``p`` [(param, coef)], ``pp``
    [(param1, param2, coef)], ``pv`` [(param, variable, coef)]; ``objective``: dict with the same lists (only its p v
    terms reach the solution: the constant of ReverseObjectiveFunction is zero).  Parameters 0-based."""
    out = []
    for c in constraints:
        kind, i = c["row"]
        cte = flat_index(n, m, p, "dh" if kind == "ineq" else "db", i)
        blk = "dG" if kind == "ineq" else "dA"
        for (prm, coef) in c.get("p", []):                        # coef * grad_cte, grad_cte = -dh_i / -db_i  (:349-360)
            out.append((prm, cte, -coef))
        for (p1, p2, coef) in c.get("pp", []):                    # :410-430 (a squared parameter lands once: both reads
            out.append((p1, cte, -coef * param_values[p2]))       #  happen before either write)
            if p2 != p1:
                out.append((p2, cte, -coef * param_values[p1]))
        for (prm, v, coef) in c.get("pv", []):                    # coef * coefficient(grad_pf, v)  (:431-437)
            out.append((prm, flat_index(n, m, p, blk, i, v), coef))
    if objective is not None:
        for (prm, v, coef) in objective.get("pv", []):            # :513-518
            out.append((prm, flat_index(n, m, p, "dq", v), coef))
    return out
