"""Synthetic, already-solved problem generators for the BASELINE.json configs (SURVEY.md §8d).

Problems are built *from* their solution (no HiGHS/Ipopt/SCS run, the primal solve is excluded
from timing anyway): pick (z, lam, nu) and data, then set h, b, q so that the KKT conditions hold
exactly.  Shared by tests/ and bench.py; no oracle or reference code involved.
"""
from __future__ import annotations

import numpy as np


def qp_batch(B, n=64, m=64, p=16, n_active=16, seed0=2026, shared=False):
    """Config 2: dense random QPs with strict complementarity and LICQ (n_active + p <= n).

    Per instance b (``default_rng(seed0 + b)``): Q = L L'/n + 0.1 I, G, A ~ N(0,1), z ~ N(0,1),
    ``n_active`` random inequality rows active (lam ~ U(.5,1.5), slack 0), the rest inactive
    (lam = 0, slack = -U(.5,1.5)), nu ~ N(0,1); h = Gz - slack, b = Az, q = -(Qz + G'lam + A'nu).
    Returns logical arrays (B, rows, cols) plus a dense forward direction and a reverse seed.
    ``shared=True``: Q, G, A identical across the batch (OptNet layer with shared weights).
    """
    d = {k: np.empty(s) for k, s in dict(
        Q=(B, n, n), G=(B, m, n), A=(B, p, n), h=(B, m), b=(B, p), q=(B, n), z=(B, n), lam=(B, m), nu=(B, p),
        dQ=(B, n, n), dq=(B, n), dG=(B, m, n), dh=(B, m), dA=(B, p, n), db=(B, p), seed=(B, n)).items()}
    for i in range(B):
        rng = np.random.default_rng(seed0 + (0 if shared else i))
        L = rng.standard_normal((n, n))
        Q = L @ L.T / n + 0.1 * np.eye(n)
        G = rng.standard_normal((m, n))
        A = rng.standard_normal((p, n))
        if shared:
            rng = np.random.default_rng(seed0 + 7919 * (i + 1))
        z = rng.standard_normal(n)
        act = rng.permutation(m)[:n_active]
        lam = np.zeros(m)
        lam[act] = rng.uniform(0.5, 1.5, size=act.size)
        slack = -rng.uniform(0.5, 1.5, size=m)
        slack[act] = 0.0
        nu = rng.standard_normal(p)
        d["Q"][i], d["G"][i], d["A"][i] = Q, G, A
        d["z"][i], d["lam"][i], d["nu"][i] = z, lam, nu
        d["h"][i] = G @ z - slack
        d["b"][i] = A @ z
        d["q"][i] = -(Q @ z + G.T @ lam + A.T @ nu)
        S = rng.standard_normal((n, n))
        d["dQ"][i] = (S + S.T) / 2
        d["dq"][i] = rng.standard_normal(n)
        d["dG"][i] = rng.standard_normal((m, n))
        d["dh"][i] = rng.standard_normal(m)
        d["dA"][i] = rng.standard_normal((p, n))
        d["db"][i] = rng.standard_normal(p)
        d["seed"][i] = rng.standard_normal(n)
    return d


def qp_batch_fast(B, n=64, m=64, p=16, n_active=16, seed=2026):
    """Same distribution as ``qp_batch`` drawn with ONE vectorised generator (for the full 4096
    batch in bench.py, where per-instance seeding only costs time)."""
    rng = np.random.default_rng(seed)
    L = rng.standard_normal((B, n, n))
    Q = L @ L.transpose(0, 2, 1) / n + 0.1 * np.eye(n)
    G = rng.standard_normal((B, m, n))
    A = rng.standard_normal((B, p, n))
    z = rng.standard_normal((B, n))
    order = np.argsort(rng.random((B, m)), axis=1)
    active = np.zeros((B, m), dtype=bool)
    np.put_along_axis(active, order[:, :n_active], True, axis=1)
    lam = np.where(active, rng.uniform(0.5, 1.5, size=(B, m)), 0.0)
    slack = np.where(active, 0.0, -rng.uniform(0.5, 1.5, size=(B, m)))
    nu = rng.standard_normal((B, p))
    h = np.einsum("bij,bj->bi", G, z) - slack
    b = np.einsum("bij,bj->bi", A, z)
    q = -(np.einsum("bij,bj->bi", Q, z) + np.einsum("bij,bi->bj", G, lam) + np.einsum("bij,bi->bj", A, nu))
    S = rng.standard_normal((B, n, n))
    return dict(Q=Q, G=G, A=A, h=h, b=b, q=q, z=z, lam=lam, nu=nu, dQ=(S + S.transpose(0, 2, 1)) / 2,
                dq=rng.standard_normal((B, n)), dG=rng.standard_normal((B, m, n)), dh=rng.standard_normal((B, m)),
                dA=rng.standard_normal((B, p, n)), db=rng.standard_normal((B, p)),
                seed=rng.standard_normal((B, n)))


def qp_batch_shared_fast(B, n=64, m=64, p=16, n_active=16, seed=4242):
    """OptNet-shared variant of config 2 (SURVEY.md 8d): ONE (Q, G, A) for the whole batch, per-instance (z, lam, nu) with
    h = G z - slack, b = A z, q = -(Q z + G'lam + A'nu): every instance is an exact KKT point of the shared matrices.
    Returns Q (n, n), G (m, n), A (p, n) and per-instance h, z, lam, nu, seed."""
    rng = np.random.default_rng(seed)
    L = rng.standard_normal((n, n))
    Q = L @ L.T / n + 0.1 * np.eye(n)
    G = rng.standard_normal((m, n))
    A = rng.standard_normal((p, n))
    z = rng.standard_normal((B, n))
    order = np.argsort(rng.random((B, m)), axis=1)
    active = np.zeros((B, m), dtype=bool)
    np.put_along_axis(active, order[:, :n_active], True, axis=1)
    lam = np.where(active, rng.uniform(0.5, 1.5, size=(B, m)), 0.0)
    slack = np.where(active, 0.0, -rng.uniform(0.5, 1.5, size=(B, m)))
    nu = rng.standard_normal((B, p))
    return dict(Q=Q, G=G, A=A, h=z @ G.T - slack, b=z @ A.T, z=z, lam=lam, nu=nu, seed=rng.standard_normal((B, n)))


def lp_config1(n=200, m=100, n_active=60, seed=1):
    """Config 1: random LP, Q == 0 -> the reference's LSQR-on-KKT branch.  Vertex-like solution:
    ``n_active`` active rows; K = [0 G'L; G D] is rank deficient by design (min-norm answer)."""
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((m, n))
    z = rng.standard_normal(n)
    act = rng.permutation(m)[:n_active]
    lam = np.zeros(m)
    lam[act] = rng.uniform(0.5, 1.5, size=n_active)
    slack = -rng.uniform(0.5, 1.5, size=m)
    slack[act] = 0.0
    return dict(Q=np.zeros((n, n)), q=-(G.T @ lam), G=G, h=G @ z - slack, A=np.zeros((0, n)), b=np.zeros(0),
                z=z, lam=lam, nu=np.zeros(0), seed=rng.standard_normal(n))


def conic_config4(n=5000, n_zero=500, n_nonneg=4000, n_soc=300, soc_dim=10, nnz_per_row=10, seed=4, psd_sides=(),
                  col_window=None, active_frac=None, solution_scale=1.0):
    """Config 4: sparse conic program solved by construction (Moreau decomposition):
    zeta ~ N(0,1)^m, s = Pi_K(zeta), y = s - zeta in K*, x ~ N(0,1)^n, b = A x + s, c = -A'y,
    so v = y - s = -zeta.  Returns A (scipy CSC, the reference's A = -coefficients), b, c, x, s, y,
    cone lists and a reverse seed.

    ``active_frac`` / ``solution_scale`` give the WELL-CONDITIONED variant used for converged parity checks: with
    zeta ~ N(0,1) half of the nonnegative rows are active and zeros + active rows + SOC rows barely exceed n, so M
    is close to singular (cond ~ 1e7; default-tolerance LSQR stops after ~1e4 iterations at a rounding-dependent
    point).  ``active_frac=0.75`` makes that fraction of the nonnegative rows active (sign of zeta chosen, magnitude
    kept) and ``solution_scale=0.02`` scales (x, s, y) so that |b|, |c| are of the order of |A| -- cond(M) ~ 1e4,
    LSQR converges in ~1e3 iterations at the default tolerances."""
    import scipy.sparse as sp
    from oracle import cones as oc  # projection only used to *construct* the data set
    rng = np.random.default_rng(seed)
    cone_types = [oc.ZERO] * (1 if n_zero else 0) + [oc.NONNEG] * (1 if n_nonneg else 0) + [oc.SOC] * n_soc + \
        [oc.PSD] * len(psd_sides)
    cone_dims = ([n_zero] if n_zero else []) + ([n_nonneg] if n_nonneg else []) + [soc_dim] * n_soc + \
        [d * (d + 1) // 2 for d in psd_sides]
    m = int(sum(cone_dims))
    rows = np.repeat(np.arange(m), nnz_per_row)
    if col_window is None:      # SURVEY 8(d): uniformly random columns
        cols = rng.integers(0, n, size=m * nnz_per_row)
    else:                       # stage-structured variant: row i touches variables within +-col_window of i n / m
        centre = (rows.astype(np.int64) * n) // m
        cols = (centre + rng.integers(-col_window, col_window + 1, size=m * nnz_per_row)) % n
    vals = rng.standard_normal(m * nnz_per_row)
    A = sp.csc_matrix((vals, (rows, cols)), shape=(m, n))
    A.sum_duplicates()
    A.sort_indices()
    zeta = rng.standard_normal(m)
    if active_frac is not None and n_nonneg:
        lo = n_zero
        act = rng.permutation(n_nonneg) < int(round(active_frac * n_nonneg))
        zeta[lo:lo + n_nonneg] = np.abs(zeta[lo:lo + n_nonneg]) * np.where(act, -1.0, 1.0)   # zeta < 0: s = 0, y > 0
    zeta *= solution_scale
    # primal cone K = product of the MOI sets; s = Pi_K(zeta).  oracle.cones projects on the DUAL of
    # the listed set, which equals the set itself for nonneg/SOC/PSD; for Zeros, K = {0}.
    s = np.empty(m)
    off = oc.cone_offsets(cone_dims)
    for k, t in enumerate(cone_types):
        sl = slice(off[k], off[k + 1])
        s[sl] = 0.0 if t == oc.ZERO else oc.project(zeta[sl], t)
    y = s - zeta
    x = rng.standard_normal(n) * solution_scale
    return dict(A=A, b=A @ x + s, c=-(A.T @ y), x=x, s=s, y=y, cone_types=cone_types, cone_dims=cone_dims,
                seed=rng.standard_normal(n))


def conic_exp_problem(n=5000, n_zero=500, n_nonneg=4000, n_soc=0, soc_dim=10, n_exp=500, n_dual_exp=500, nnz_per_row=10,
                      seed=7, psd_sides=(), solution_scale=1.0, n_pow=0, n_dual_pow=0):
    """Config-4-like sparse conic program with ``n_exp`` ExponentialCone and ``n_dual_exp`` DualExponentialCone
    constraints (3 rows each) after the zero, nonnegative and SOC rows (and PSD cones, if any), then ``n_pow`` PowerCone
    and ``n_dual_pow`` DualPowerCone constraints (3 rows each), solved by construction like ``conic_config4``:
    zeta ~ N(0,1)^m, s = Pi_K(zeta) onto the primal cone K (the listed sets), y = s - zeta in K*, b = A x + s,
    c = -A'y.  The exponential and power cones are not self-dual: pow_cone_oracle.project(., t) projects onto the DUAL
    of set t, so the primal projection of an EXP slice is project(., DUAL_EXP) and vice versa (POW likewise).  Every
    third exp / power slice is drawn with |zeta| mixed in scale so that all curved-cone cases occur.  The power cones'
    exponents (uniform in [0.05, 0.95]), their order and scales come from a second generator seeded from ``seed``, so
    the data without power cones is what it always was.  ``cone_params`` holds each cone's exponent (0 for the other
    cones)."""
    import scipy.sparse as sp

    import pow_cone_oracle as oc  # projection only used to *construct* the data set
    rng = np.random.default_rng(seed)
    prng = np.random.default_rng([seed, 6])
    cone_types = [oc.ZERO] * (1 if n_zero else 0) + [oc.NONNEG] * (1 if n_nonneg else 0) + [oc.SOC] * n_soc + \
        [oc.PSD] * len(psd_sides)
    cone_dims = ([n_zero] if n_zero else []) + ([n_nonneg] if n_nonneg else []) + [soc_dim] * n_soc + \
        [d * (d + 1) // 2 for d in psd_sides]
    kinds = np.array([oc.EXP] * n_exp + [oc.DUAL_EXP] * n_dual_exp)
    kinds = kinds[rng.permutation(kinds.size)]
    cone_types += kinds.tolist()
    cone_dims += [3] * kinds.size
    cone_params = [0.0] * len(cone_types)
    if n_pow or n_dual_pow:
        pkinds = np.array([oc.POW] * n_pow + [oc.DUAL_POW] * n_dual_pow)
        pkinds = pkinds[prng.permutation(pkinds.size)]
        cone_types += pkinds.tolist()
        cone_dims += [3] * pkinds.size
        cone_params += prng.uniform(0.05, 0.95, pkinds.size).tolist()
    m = int(sum(cone_dims))
    rows = np.repeat(np.arange(m), nnz_per_row)
    cols = rng.integers(0, n, size=m * nnz_per_row)
    A = sp.csc_matrix((rng.standard_normal(m * nnz_per_row), (rows, cols)), shape=(m, n))
    A.sum_duplicates()
    A.sort_indices()
    zeta = rng.standard_normal(m)
    off = oc.cone_offsets(cone_dims)
    for k, t in enumerate(cone_types):
        if t in (oc.EXP, oc.DUAL_EXP) and k % 3 == 0:
            zeta[off[k]:off[k + 1]] *= 10.0 ** rng.uniform(-1, 1, 3)
        elif t in (oc.POW, oc.DUAL_POW) and k % 3 == 0:
            zeta[off[k]:off[k + 1]] *= 10.0 ** prng.uniform(-1, 1, 3)
    zeta *= solution_scale
    dual_of = {oc.EXP: oc.DUAL_EXP, oc.DUAL_EXP: oc.EXP, oc.POW: oc.DUAL_POW, oc.DUAL_POW: oc.POW}
    s = np.empty(m)
    for k, t in enumerate(cone_types):
        sl = slice(off[k], off[k + 1])
        s[sl] = 0.0 if t == oc.ZERO else oc.project(zeta[sl], dual_of.get(t, t), cone_params[k])
    y = s - zeta
    x = rng.standard_normal(n) * solution_scale
    return dict(A=A, b=A @ x + s, c=-(A.T @ y), x=x, s=s, y=y, cone_types=cone_types, cone_dims=cone_dims,
                cone_params=cone_params, seed=rng.standard_normal(n))


def conic_config4_conditioned(**kw):
    """Config 4 with 75 % of the nonnegative rows active and the solution scaled by 0.02 (see ``conic_config4``)."""
    kw.setdefault("active_frac", 0.75)
    kw.setdefault("solution_scale", 0.02)
    return conic_config4(**kw)


def mpc_config3(T=10_000, nx=6, nu=4, active_frac=0.1, seed=3):
    """Config 3: one sparse MPC QP, solved by construction.  Stage t = 0..T-1 has state x_t (nx) and input u_t (nu);
    z = (x_0, u_0, x_1, u_1, ...), n = T (nx + nu).  Q = blkdiag(Qx, R) per stage (SPD); dynamics equalities
    x_{t+1} = Ad x_t + Bd u_t (x_0 fixed: nx rows), p = T nx; input box constraints -1 <= u <= 1 as 2 nu rows per
    stage, m = 2 T nu, a fraction ``active_frac`` of the inputs sits on a bound (lam > 0, slack 0), the others are
    strictly inside (lam = 0).  Returns the reference's LHS (scipy CSC, create_LHS_matrix layout) and the pieces."""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    n, p, m = T * (nx + nu), T * nx, 2 * T * nu
    Lx = rng.standard_normal((nx, nx)); Qx = Lx @ Lx.T / nx + 0.5 * np.eye(nx)
    Lr = rng.standard_normal((nu, nu)); R = Lr @ Lr.T / nu + 0.5 * np.eye(nu)
    Ad = rng.standard_normal((nx, nx)) / np.sqrt(nx)
    Ad *= 0.95 / np.abs(np.linalg.eigvals(Ad)).max()
    Bd = rng.standard_normal((nx, nu)) / np.sqrt(nx)
    Q = sp.block_diag([sp.csc_matrix(np.block([[Qx, np.zeros((nx, nu))], [np.zeros((nu, nx)), R]]))] * T, format="csc")
    # equality rows: block t couples stage t-1 (Ad, Bd) and x_t (-I); block 0 is x_0 = given
    rows, cols, vals = [], [], []
    s = nx + nu
    for t in range(T):
        r0 = t * nx
        for i in range(nx):
            rows.append(r0 + i); cols.append(t * s + i); vals.append(-1.0)
        if t > 0:
            c0 = (t - 1) * s
            rr, cc = np.meshgrid(np.arange(nx), np.arange(nx), indexing="ij")
            rows += list(r0 + rr.ravel()); cols += list(c0 + cc.ravel()); vals += list(Ad.ravel())
            rr, cc = np.meshgrid(np.arange(nx), np.arange(nu), indexing="ij")
            rows += list(r0 + rr.ravel()); cols += list(c0 + nx + cc.ravel()); vals += list(Bd.ravel())
    A = sp.csc_matrix((vals, (rows, cols)), shape=(p, n))
    # inequality rows: for every input, u <= 1 and -u <= 1
    ucols = (np.arange(T)[:, None] * s + nx + np.arange(nu)[None, :]).ravel()
    G = sp.vstack([sp.csc_matrix((np.ones(T * nu), (np.arange(T * nu), ucols)), shape=(T * nu, n)),
                   sp.csc_matrix((-np.ones(T * nu), (np.arange(T * nu), ucols)), shape=(T * nu, n))]).tocsc()
    z = rng.standard_normal(n) * 0.3
    u = rng.uniform(-0.9, 0.9, size=T * nu)
    act = rng.random(T * nu) < active_frac
    side = rng.random(T * nu) < 0.5
    u[act & side] = 1.0
    u[act & ~side] = -1.0
    z[ucols] = u
    lam = np.zeros(m)
    lam[:T * nu][act & side] = rng.uniform(0.5, 1.5, size=int((act & side).sum()))
    lam[T * nu:][act & ~side] = rng.uniform(0.5, 1.5, size=int((act & ~side).sum()))
    h = np.ones(m)
    D = G @ z - h                                   # exactly 0 on the active rows, < 0 elsewhere
    nu_ = rng.standard_normal(p)
    K = sp.bmat([[Q, G.T @ sp.diags(lam), A.T], [G, sp.diags(D), None], [A, None, sp.csc_matrix((p, p))]], format="csc")
    K.sort_indices()
    return dict(K=K, Q=Q, G=G, A=A, z=z, lam=lam, nu=nu_, h=h, n=n, m=m, p=p)


def maxcut_config5(d=200, r=20, seed=5):  # r(r+1)/2 <= d makes the pair nondegenerate (unique dual): r <= 19 at d = 200
    """Config 5: max-cut SDP relaxation with a d x d PSD cone, solved by construction.  V ~ N(0,1)^{d x r} with unit
    rows, X = V V' (unit diagonal, rank r); W = orthonormal basis of range(V)^perp, S = W diag(U(.5,1.5)) W';
    nu ~ N(0,1)^d; C = S + Diag(nu): a strictly complementary primal-dual pair.  Variables = triangle of X
    (unscaled, column-wise upper), rows = Zeros(d) (X_ii = 1) + PSD triangle.  Returns A (the reference's
    A = -coefficients), b, c, x, s, y, cone lists and a reverse seed."""
    import scipy.sparse as sp
    from oracle import cones as oc  # vec_symm only: used to *construct* the data set
    rng = np.random.default_rng(seed)
    V = rng.normal(size=(d, r))
    V /= np.linalg.norm(V, axis=1, keepdims=True)
    X = V @ V.T
    Qf, _ = np.linalg.qr(np.hstack([V, rng.normal(size=(d, d - r))]))
    W = Qf[:, r:]
    S = (W * rng.uniform(0.5, 1.5, size=d - r)) @ W.T
    k = d * (d + 1) // 2
    s = np.concatenate([np.zeros(d), oc.vec_symm(X)])
    y = np.concatenate([rng.normal(size=d), oc.vec_symm(S)])
    iu = [(i * (i + 1) // 2 + i) for i in range(d)]
    A = sp.vstack([sp.csc_matrix((np.ones(d), (np.arange(d), iu)), shape=(d, k)), -sp.identity(k)]).tocsc()
    x = oc.vec_symm(X)
    return dict(A=A, b=A @ x + s, c=-(A.T @ y), x=x, s=s, y=y, cone_types=[oc.ZERO, oc.PSD], cone_dims=[d, k],
                seed=rng.normal(size=k), X=X, S=S, d=d)


def portfolio_config3(n=100_000, nfac=100, density=0.1, active_frac=0.3, seed=33):
    """Config 3, portfolio variant: n assets, ``nfac`` factors, Q = D + F F' in lifted sparse form (variables (x, y) with
    the equalities F'x - y = 0), one budget equality 1'x = 1, long-only bounds x >= 0.  z = (x, y), n + nfac
    variables; m = n inequality rows (-x <= 0), p = nfac + 1 equality rows.  ``active_frac`` of the assets sit on the
    bound (x = 0, lam > 0).  The KKT pattern is an arrowhead: every asset couples to the dense budget row and to the
    factor rows it loads on -- not banded under any ordering.  Returns the reference's LHS (create_LHS_matrix)."""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    nv = n + nfac
    F = sp.random(n, nfac, density=density, random_state=np.random.RandomState(seed), format="csc",
                  data_rvs=lambda k: rng.standard_normal(k))
    D = rng.uniform(0.5, 1.5, size=n)
    Q = sp.diags(np.concatenate([D, np.ones(nfac)]), format="csc")
    A = sp.vstack([sp.hstack([F.T, -sp.identity(nfac)]), sp.hstack([sp.csr_matrix(np.ones((1, n))), sp.csr_matrix((1, nfac))])]).tocsc()
    G = sp.hstack([-sp.identity(n), sp.csc_matrix((n, nfac))]).tocsc()
    act = rng.random(n) < active_frac
    x = np.where(act, 0.0, rng.uniform(0.1, 1.0, size=n))
    x /= x.sum()
    z = np.concatenate([x, F.T @ x])
    lam = np.where(act, rng.uniform(0.5, 1.5, size=n), 0.0)
    nu = rng.standard_normal(nfac + 1)
    h = np.zeros(n)
    Dg = G @ z - h
    K = sp.bmat([[Q, G.T @ sp.diags(lam), A.T], [G, sp.diags(Dg), None], [A, None, sp.csc_matrix((nfac + 1, nfac + 1))]], format="csc")
    K.sort_indices()
    return dict(K=K, Q=Q, G=G, A=A, z=z, lam=lam, nu=nu, h=h, n=nv, m=n, p=nfac + 1)
