# DiffOptB200.jl -- Julia host side of the B200 sensitivity hot path (thin `ccall` layer over
# include/diffopt_b200.h).  NOT executed in the build image (no Julia there); it is the binding a
# DiffOpt.jl maintainer adds, kept in sync with the C header and exercised through the identical C ABI
# by the Python ctypes mirror in diffopt.jl_b200/ (see INTEGRATION.md).
#
# Plug points used (reference tree andrewrosemberg/DiffOpt.jl v0.5.0):
#   * DiffOpt.ModelConstructor            src/moi_wrapper.jl:504-514, consumed by _diff :619-657
#   * QuadraticProgram.LinearAlgebraSolver + solve_system(solver, LHS, RHS, iterative)
#                                         src/QuadraticProgram/QuadraticProgram.jl:476-502
module DiffOptB200

import DiffOpt
import LinearAlgebra
import MathOptInterface as MOI
import SparseArrays

const LIB = get(ENV, "DIFFOPT_B200_LIB", "libdiffopt_b200")
const HOST = Cint(0)
const DEVICE = Cint(1)

struct B200Error <: Exception
    code::Int32
    msg::String
end

mutable struct Context
    handle::Ptr{Cvoid}
    function Context(device::Integer = 0)
        ref = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:diffopt_b200_create, LIB), Int32, (Int32, Ptr{Ptr{Cvoid}}), device, ref)
        rc == 0 || throw(B200Error(rc, "diffopt_b200_create failed (no B200 / no CUDA device: there is no CPU fallback)"))
        ctx = new(ref[])
        finalizer(c -> ccall((:diffopt_b200_destroy, LIB), Int32, (Ptr{Cvoid},), c.handle), ctx)
        return ctx
    end
end

last_error(ctx::Context) = unsafe_string(ccall((:diffopt_b200_last_error, LIB), Cstring, (Ptr{Cvoid},), ctx.handle))

# rc < 0: bad argument / CUDA error -> error(...) like the reference's generic failures;
# rc > 0: LAPACK-style info -> SingularException, what `LHS \ RHS` throws in the reference.
function check(ctx::Context, rc::Int32)
    rc < 0 && throw(B200Error(rc, last_error(ctx)))
    rc > 0 && throw(LinearAlgebra.SingularException(Int(rc)))
    return
end

# ------------------------------------------------------------------------------------------------
# (1) Narrow plug point: a linear solver for QuadraticProgram.Model
#     model.linear_solver = B200Solver(ctx);  solve_system is called from
#     reverse_differentiate! (:335, LHS) and forward_differentiate! (:438, LHS')
# ------------------------------------------------------------------------------------------------
struct B200Solver
    ctx::Context
    atol::Float64
    btol::Float64
    conlim::Float64
end
B200Solver(ctx::Context) = B200Solver(ctx, sqrt(eps()), sqrt(eps()), 1 / sqrt(eps()))  # IterativeSolvers.lsqr defaults

_csc(A::SparseArrays.SparseMatrixCSC{Float64,Int}) = (A, Cint(0))
_csc(A::LinearAlgebra.Adjoint{Float64,<:SparseArrays.SparseMatrixCSC{Float64,Int}}) = (parent(A), Cint(1))

function DiffOpt.QuadraticProgram.solve_system(s::B200Solver, LHS, RHS::AbstractVector, iterative::Bool)
    A, trans = _csc(LHS)
    rhs = Vector{Float64}(RHS)           # forward mode may hand over a SparseVector (:493-496)
    n = size(A, 1)
    x = Vector{Float64}(undef, n)
    GC.@preserve A rhs x begin
        rc = if iterative
            # LP branch: IterativeSolvers.lsqr(LHS, RHS) -> persistent device LSQR on the CSC matrix
            ccall((:diffopt_b200_lsqr_csc, LIB), Int32,
                  (Ptr{Cvoid}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int32, Ptr{Float64},
                   Float64, Float64, Float64, Int64, Ptr{Float64}, Ptr{Float64}, Int32),
                  s.ctx.handle, size(A, 1), size(A, 2), A.colptr, A.rowval, A.nzval, trans, rhs,
                  s.atol, s.btol, s.conlim, max(size(A)...), x, C_NULL, HOST)
        else
            # `LHS \ RHS`: pivoted LU on the device (dense kernel up to N = 1024, multifrontal sparse LU beyond)
            ccall((:diffopt_b200_kkt_solve_csc, LIB), Int32,
                  (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int32, Int64, Ptr{Float64}, Ptr{Float64}, Int32),
                  s.ctx.handle, n, A.colptr, A.rowval, A.nzval, trans, 1, rhs, x, HOST)
        end
    end
    check(s.ctx, rc)
    return x
end

"""
    SparseFactorization(ctx, LHS)            # LHS::SparseMatrixCSC or its Adjoint

One device factorisation of a large sparse KKT matrix (multifrontal LU: nested dissection + partial pivoting inside the
fronts), reused for any number of right-hand sides: `F \\ RHS` with `RHS::Matrix` (N x nrhs).  Replaces the per-direction `LHS' \\ RHS` of
`forward_differentiate!` (QuadraticProgram.jl:438) when many directions are differentiated against one solution.
"""
struct SparseFactorization
    ctx::Context
    n::Int
    function SparseFactorization(ctx::Context, LHS)
        A, trans = _csc(LHS)
        GC.@preserve A begin
            rc = ccall((:diffopt_b200_sparse_setup, LIB), Int32,
                       (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int32, Ptr{Int64}),
                       ctx.handle, size(A, 1), A.colptr, A.rowval, A.nzval, trans, C_NULL)
        end
        check(ctx, rc)
        return new(ctx, size(A, 1))
    end
end

function Base.:\(F::SparseFactorization, RHS::StridedVecOrMat{Float64})
    X = similar(RHS)
    GC.@preserve RHS X begin
        rc = ccall((:diffopt_b200_sparse_solve, LIB), Int32, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Int32),
                   F.ctx.handle, size(RHS, 2), RHS, X, HOST)
    end
    check(F.ctx, rc)
    return X
end

"ModelConstructor that keeps the B200 solver attached although the wrapper rebuilds the backend (moi_wrapper.jl:619-657)."
function qp_model_constructor(ctx::Context)
    return () -> begin
        m = DiffOpt.QuadraticProgram.Model()
        m.linear_solver = B200Solver(ctx)
        m
    end
end
# usage:  MOI.set(model, DiffOpt.ModelConstructor(), DiffOptB200.qp_model_constructor(ctx))

# Process-wide default context (device from ENV["DIFFOPT_B200_DEVICE"], default 0) for the zero-argument constructors
# that `DiffOpt.ModelConstructor` needs (`MOI.instantiate(ctor)` calls it without arguments, moi_wrapper.jl:619-657).
const _DEFAULT_CTX = Ref{Union{Nothing,Context}}(nothing)
function default_context()
    if _DEFAULT_CTX[] === nothing
        _DEFAULT_CTX[] = Context(parse(Int, get(ENV, "DIFFOPT_B200_DEVICE", "0")))
    end
    return _DEFAULT_CTX[]::Context
end

"""
    DiffOptB200.QPModel()

Backend for `MOI.set(model, DiffOpt.ModelConstructor(), DiffOptB200.QPModel)`: the reference's own
`DiffOpt.QuadraticProgram.Model` (a `DiffOpt.AbstractModel`; all of its MOI plumbing, caches and getters are kept as
they are, QuadraticProgram.jl:60-473) with its linear algebra -- the only part that costs time,
`solve_system` at :335 and :438 -- bound to the GPU through `B200Solver`.
"""
QPModel() = qp_model_constructor(default_context())()

# ------------------------------------------------------------------------------------------------
# (2) Batched QP sensitivities (OptNet-style layers): B independent instances, dense column-major
#     arrays exactly as Julia stores them: Q[n,n,B], G[m,n,B], A[p,n,B], h[m,B], z[n,B], lam[m,B], nu[p,B]
#     (lam, nu are the reference's stored duals, i.e. NEGATED MOI duals, QuadraticProgram.jl:156-180).
#     One call = create_LHS_matrix (:256-282) + forward (:357-446) + reverse (:316-351) for every instance.
# ------------------------------------------------------------------------------------------------
_p(a::Nothing) = Ptr{Float64}(C_NULL)
_p(a::Array{Float64}) = pointer(a)

function qp_batch_solve(ctx::Context, Q, G, A, h, z, lam, nu;
                        dQ = nothing, dq = nothing, dG = nothing, dh = nothing, dA = nothing, db = nothing,
                        dl_dz = nothing)
    n, B = size(z)
    m = size(lam, 1)
    p = size(nu, 1)
    N = n + m + p
    fwd = any(!isnothing, (dQ, dq, dG, dh, dA, db)) ? Matrix{Float64}(undef, N, B) : nothing
    rev = dl_dz === nothing ? nothing : Matrix{Float64}(undef, N, B)
    info = zeros(Int32, B)
    GC.@preserve Q G A h z lam nu dQ dq dG dh dA db dl_dz fwd rev info begin
        rc = ccall((:diffopt_b200_qp_batch_solve, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Int32, Int32, Int32,
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                    Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Int32),
                   ctx.handle, B, n, m, p, _p(Q), _p(G), _p(A), _p(h), _p(z), _p(lam), _p(nu),
                   _p(dQ), _p(dq), _p(dG), _p(dh), _p(dA), _p(db), _p(dl_dz), _p(fwd), _p(rev), info, HOST)
    end
    check(ctx, rc)
    split(x) = x === nothing ? nothing : (dz = x[1:n, :], dλ = x[n+1:n+m, :], dν = x[n+m+1:end, :])
    return (forward = split(fwd), reverse = split(rev), info = info)
end

"""
    qp_batch_solve_lsqr(ctx, G, A, h, z, lam, nu; dQ, dq, dG, dh, dA, db, dl_dz, shared_matrices, atol, btol, conlim, maxiter)

The LSQR branch of `solve_system` (Q = 0, QuadraticProgram.jl:486-488) for a batch of LPs, one CTA per instance: singular
KKT matrices give LSQR's minimum-norm answer as in the reference.  Layouts as `qp_batch_solve` without Q (`G` of size
(m, n, B), or (m, n) with `shared_matrices = true`).  Tolerances default to IterativeSolvers' values; `maxiter = 0` means
n + m + p.  `stats[:, k, b]` = (istop, itn, rnorm, arnorm) of the forward (k = 1) and reverse (k = 2) solve of instance b.
"""
function qp_batch_solve_lsqr(ctx::Context, G, A, h, z, lam, nu;
                             dQ = nothing, dq = nothing, dG = nothing, dh = nothing, dA = nothing, db = nothing,
                             dl_dz = nothing, shared_matrices::Bool = false, atol::Float64 = sqrt(eps(Float64)),
                             btol::Float64 = sqrt(eps(Float64)), conlim::Float64 = 1 / sqrt(eps(Float64)),
                             maxiter::Integer = 0)
    n, B = size(z)
    m = size(lam, 1)
    p = size(nu, 1)
    N = n + m + p
    fwd = any(!isnothing, (dQ, dq, dG, dh, dA, db)) ? Matrix{Float64}(undef, N, B) : nothing
    rev = dl_dz === nothing ? nothing : Matrix{Float64}(undef, N, B)
    stats = zeros(Float64, 4, 2, B)
    GC.@preserve G A h z lam nu dQ dq dG dh dA db dl_dz fwd rev stats begin
        rc = ccall((:diffopt_b200_qp_batch_solve_lsqr, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Int32, Int32, Int32,
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                    Float64, Float64, Float64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Int32),
                   ctx.handle, B, n, m, p, _p(G), _p(A), _p(h), _p(z), _p(lam), _p(nu),
                   _p(dQ), _p(dq), _p(dG), _p(dh), _p(dA), _p(db), _p(dl_dz), atol, btol, conlim, maxiter,
                   _p(fwd), _p(rev), stats, HOST, shared_matrices ? QP_SHARED_MATRICES : Int32(0))
    end
    check(ctx, rc)
    split(x) = x === nothing ? nothing : (dz = x[1:n, :], dλ = x[n+1:n+m, :], dν = x[n+m+1:end, :])
    return (forward = split(fwd), reverse = split(rev), stats = stats)
end

# Stream-ordered form for device-resident batches (pointers of CUDA.jl arrays, `pointer(x)` converted to Ptr{Float64}):
# enqueue any number of batches, then `synchronize(ctx)` waits and throws for the status of the last one.
function qp_batch_solve_async(ctx::Context, B::Integer, n::Integer, m::Integer, p::Integer,
                              Q::Ptr{Float64}, G::Ptr{Float64}, A::Ptr{Float64}, h::Ptr{Float64}, z::Ptr{Float64},
                              lam::Ptr{Float64}, nu::Ptr{Float64}, dQ::Ptr{Float64}, dq::Ptr{Float64},
                              dG::Ptr{Float64}, dh::Ptr{Float64}, dA::Ptr{Float64}, db::Ptr{Float64},
                              dl_dz::Ptr{Float64}, fwd::Ptr{Float64}, rev::Ptr{Float64}, info::Ptr{Int32})
    rc = ccall((:diffopt_b200_qp_batch_solve_async, LIB), Int32,
               (Ptr{Cvoid}, Int64, Int32, Int32, Int32,
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
               ctx.handle, B, n, m, p, Q, G, A, h, z, lam, nu, dQ, dq, dG, dh, dA, db, dl_dz, fwd, rev, info)
    check(ctx, rc)
    return nothing
end

synchronize(ctx::Context) = check(ctx, ccall((:diffopt_b200_synchronize, LIB), Int32, (Ptr{Cvoid},), ctx.handle))

# Factorise once, solve many directions: setup keeps the batch resident, factorize stores every instance's LDL' factor, the
# multi calls take k directions per instance as Array{Float64,3} of size (rows, k, B) and return (N, k, B) blocks.
function qp_batch_setup(ctx::Context, Q, G, A, h, z, lam, nu)
    n, B = size(z)
    m = size(lam, 1)
    p = size(nu, 1)
    GC.@preserve Q G A h z lam nu begin
        rc = ccall((:diffopt_b200_qp_batch_setup, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Int32, Int32, Int32,
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32),
                   ctx.handle, B, n, m, p, _p(Q), _p(G), _p(A), _p(h), _p(z), _p(lam), _p(nu), HOST)
    end
    check(ctx, rc)
    return (B = B, n = n, m = m, p = p)
end

function qp_batch_factorize(ctx::Context, B::Integer)
    info = zeros(Int32, B)
    rc = ccall((:diffopt_b200_qp_batch_factorize, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}, Int32), ctx.handle, info, HOST)
    check(ctx, rc)
    return info
end

function qp_batch_reverse_multi(ctx::Context, shape, dl_dz::Array{Float64,3})
    n, k, B = size(dl_dz)
    N = shape.n + shape.m + shape.p
    rev = Array{Float64,3}(undef, N, k, B)
    GC.@preserve dl_dz rev begin
        rc = ccall((:diffopt_b200_qp_batch_reverse_multi, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Int32), ctx.handle, k, dl_dz, rev, HOST)
    end
    check(ctx, rc)
    return rev
end

# dQ, dG, dA: (ptr, I, J, V) of the B*k direction slots (0-based offsets, 1-based I, J), or nothing
struct CooBatch
    ptr::Ptr{Int64}
    I::Ptr{Int64}
    J::Ptr{Int64}
    V::Ptr{Float64}
end
_coo(t::Nothing) = nothing
_coo(t::Tuple) = Ref(CooBatch(pointer(t[1]), pointer(t[2]), pointer(t[3]), pointer(t[4])))
_cp(r::Nothing) = Ptr{CooBatch}(C_NULL)
_cp(r::Ref{CooBatch}) = Base.unsafe_convert(Ptr{CooBatch}, r)

function qp_batch_forward_multi(ctx::Context, shape, k::Integer; dQ = nothing, dq = nothing, dG = nothing, dh = nothing,
                                dA = nothing, db = nothing)
    N = shape.n + shape.m + shape.p
    fwd = Array{Float64,3}(undef, N, k, shape.B)
    cq, cg, ca = _coo(dQ), _coo(dG), _coo(dA)
    GC.@preserve dQ dq dG dh dA db cq cg ca fwd begin
        rc = ccall((:diffopt_b200_qp_batch_forward_multi, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Ptr{CooBatch}, Ptr{Float64}, Ptr{CooBatch}, Ptr{Float64}, Ptr{CooBatch}, Ptr{Float64},
                    Ptr{Float64}, Int32),
                   ctx.handle, k, _cp(cq), _p(dq), _cp(cg), _p(dh), _cp(ca), _p(db), fwd, HOST)
    end
    check(ctx, rc)
    return fwd
end

# ------------------------------------------------------------------------------------------------
# (3) ConicProgram backend: _gradient_cache / forward / reverse (src/ConicProgram/ConicProgram.jl:172-394)
#     cone_type: 0 Zeros, 1 Nonnegatives, 2 SecondOrderCone, 3 PositiveSemidefiniteConeTriangle, 4 ExponentialCone,
#     5 DualExponentialCone, 6 PowerCone, 7 DualPowerCone (row order of A); cone_param: the exponent of each power cone
# ------------------------------------------------------------------------------------------------
function conic_setup(ctx::Context, A::SparseArrays.SparseMatrixCSC{Float64,Int}, b, c, x, s, y,
                     cone_type::Vector{Int32}, cone_dim::Vector{Int64}, cone_param::Vector{Float64} = zeros(length(cone_type)))
    m, n = size(A)
    GC.@preserve A b c x s y cone_type cone_dim cone_param begin
        rc = ccall((:diffopt_b200_conic_setup_ex, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Int32}, Ptr{Int64}, Ptr{Float64}, Int32),
                   ctx.handle, n, m, A.colptr, A.rowval, A.nzval, b, c, x, s, y, length(cone_type), cone_type, cone_dim,
                   cone_param, HOST)
    end
    check(ctx, rc)
end

"reverse_differentiate! (:336-394): g = lsqr(M, [dx; 0; -x'dx]); returns (g, dc, db) with the getters of :396-428."
function conic_reverse(ctx::Context, n::Int, m::Int, dx::Vector{Float64};
                       atol = sqrt(eps()), btol = sqrt(eps()), conlim = 1 / sqrt(eps()), maxiter = n + m + 1)
    g = Vector{Float64}(undef, n + m + 1); dc = Vector{Float64}(undef, n); db = Vector{Float64}(undef, m)
    stats = zeros(4)
    GC.@preserve dx g dc db stats begin
        rc = ccall((:diffopt_b200_conic_reverse, LIB), Int32,
                   (Ptr{Cvoid}, Ptr{Float64}, Float64, Float64, Float64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32),
                   ctx.handle, dx, atol, btol, conlim, maxiter, g, dc, db, stats, HOST)
    end
    check(ctx, rc)
    return (g = g, dc = dc, db = db, istop = Int(stats[1]), iterations = Int(stats[2]))
end

"forward_differentiate! (:257-334): dA as COO triplets exactly as packed by the reference (un-negated, :296-305)."
function conic_forward(ctx::Context, n::Int, m::Int, dA_rows::Vector{Int64}, dA_cols::Vector{Int64}, dA_vals::Vector{Float64},
                       db, dc; atol = sqrt(eps()), btol = sqrt(eps()), conlim = 1 / sqrt(eps()), maxiter = n + m + 1)
    dx = Vector{Float64}(undef, n); dz = Vector{Float64}(undef, n + m + 1); stats = zeros(4)
    GC.@preserve dA_rows dA_cols dA_vals db dc dx dz stats begin
        rc = ccall((:diffopt_b200_conic_forward, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                    Float64, Float64, Float64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32),
                   ctx.handle, length(dA_vals), dA_rows, dA_cols, dA_vals, _p(db), _p(dc), atol, btol, conlim, maxiter, dx, dz, stats, HOST)
    end
    check(ctx, rc)
    return (dx = dx, dz = dz, iterations = Int(stats[2]))
end

# Many directions per call against the current conic_setup (one LSQR launch): Jacobian columns or many sensitivity
# directions.  Matrices are (rows, k): column j is direction j.  Like the QP multi helpers, these have not been run yet.
"k reverse seeds dx (n, k) -> (g (n+m+1, k), dc (n, k), db (n, k), stats (4, k)) of reverse_differentiate! (:336-394)."
function conic_reverse_multi(ctx::Context, n::Int, m::Int, dx::Matrix{Float64};
                             atol = sqrt(eps()), btol = sqrt(eps()), conlim = 1 / sqrt(eps()), maxiter = n + m + 1)
    k = size(dx, 2)
    g = Matrix{Float64}(undef, n + m + 1, k); dc = Matrix{Float64}(undef, n, k); db = Matrix{Float64}(undef, m, k)
    stats = zeros(4, k)
    GC.@preserve dx g dc db stats begin
        rc = ccall((:diffopt_b200_conic_reverse_multi, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Ptr{Float64}, Float64, Float64, Float64, Int64, Ptr{Float64}, Ptr{Float64},
                    Ptr{Float64}, Ptr{Float64}, Int32),
                   ctx.handle, k, dx, atol, btol, conlim, maxiter, g, dc, db, stats, HOST)
    end
    check(ctx, rc)
    return (g = g, dc = dc, db = db, stats = stats)
end

"k forward directions of forward_differentiate! (:257-334): dA as (ptr, I, J, V) with k+1 offsets (or nothing),
db (m, k), dc (n, k) (or nothing) -> (dx (n, k), dz (n+m+1, k), stats (4, k))."
function conic_forward_multi(ctx::Context, n::Int, m::Int, k::Integer; dA = nothing, db = nothing, dc = nothing,
                             atol = sqrt(eps()), btol = sqrt(eps()), conlim = 1 / sqrt(eps()), maxiter = n + m + 1)
    dx = Matrix{Float64}(undef, n, k); dz = Matrix{Float64}(undef, n + m + 1, k); stats = zeros(4, k)
    ca = _coo(dA)
    GC.@preserve dA db dc ca dx dz stats begin
        rc = ccall((:diffopt_b200_conic_forward_multi, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Ptr{CooBatch}, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Float64, Int64,
                    Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32),
                   ctx.handle, k, _cp(ca), _p(db), _p(dc), atol, btol, conlim, maxiter, dx, dz, stats, HOST)
    end
    check(ctx, rc)
    return (dx = dx, dz = dz, stats = stats)
end

# ------------------------------------------------------------------------------------------------
# (4) ConicModel <: DiffOpt.AbstractModel -- the conic backend behind `DiffOpt.ModelConstructor`
#     (no narrow hook exists for ConicProgram, so the backend type itself is provided).  Same stored quantities as
#     DiffOpt.ConicProgram.Model (ConicProgram.jl:78-101): the geometric-form MOI model, the input cache, x, s, y;
#     `_gradient_cache` (:172-255), the LSQR solves (:323, :372) and pi / Dpi run on the device.
#     usage:  MOI.set(model, DiffOpt.ModelConstructor(), DiffOptB200.ConicModel)
# ------------------------------------------------------------------------------------------------
const CP = DiffOpt.ConicProgram

mutable struct ConicModel <: DiffOpt.AbstractModel
    model::CP.Form{Float64}                      # constraints in matrix form (MatrixOfConstraints, ProductOfSets)
    ctx::Context
    cache_valid::Bool                            # device-side gradient cache matches (model, x, s, y)
    vp::Vector{Float64}                          # pi(y - s), fetched once per cache (getters :396-443 need it)
    forw_grad_cache::Union{Nothing,CP.ForwCache}
    back_grad_cache::Union{Nothing,CP.ReverseCache}
    input_cache::DiffOpt.InputCache
    x::Vector{Float64}
    s::Vector{Float64}
    y::Vector{Float64}
    diff_time::Float64
    lsqr_atol::Float64
    lsqr_btol::Float64
    lsqr_conlim::Float64
end

function ConicModel(ctx::Context = default_context())
    return ConicModel(CP.Form{Float64}(), ctx, false, Float64[], nothing, nothing, DiffOpt.InputCache(),
                      Float64[], Float64[], Float64[], NaN, sqrt(eps()), sqrt(eps()), 1 / sqrt(eps()))
end

MOI.is_empty(model::ConicModel) = MOI.is_empty(model.model)

function MOI.empty!(model::ConicModel)
    MOI.empty!(model.model)
    model.cache_valid = false
    model.forw_grad_cache = nothing
    model.back_grad_cache = nothing
    empty!(model.input_cache)
    empty!(model.x); empty!(model.s); empty!(model.y); empty!(model.vp)
    model.diff_time = NaN
    return
end

MOI.get(model::ConicModel, ::DiffOpt.DifferentiateTimeSec) = model.diff_time

# set types are registered in the ProductOfSets on first sight, as ConicProgram.jl:132-142 does
function MOI.supports_constraint(model::ConicModel, F::Type{MOI.VectorAffineFunction{Float64}},
                                 ::Type{S}) where {S<:MOI.AbstractVectorSet}
    if DiffOpt.add_set_types(model.model.constraints.sets, S)
        push!(model.model.constraints.caches, Tuple{F,S}[])
        push!(model.model.constraints.are_indices_mapped, BitSet())
    end
    return MOI.supports_constraint(model.model, F, S)
end

function MOI.set(model::ConicModel, ::MOI.ConstraintPrimalStart, ci::MOI.ConstraintIndex, value)
    MOI.throw_if_not_valid(model, ci)
    model.cache_valid = false
    return DiffOpt._enlarge_set(model.s, MOI.Utilities.rows(model.model.constraints, ci), value)
end

function MOI.set(model::ConicModel, ::MOI.ConstraintDualStart, ci::MOI.ConstraintIndex, value)
    MOI.throw_if_not_valid(model, ci)
    model.cache_valid = false
    return DiffOpt._enlarge_set(model.y, MOI.Utilities.rows(model.model.constraints, ci), value)
end

_cone_code(::Type{MOI.Zeros}) = Int32(0)
_cone_code(::Type{MOI.Nonnegatives}) = Int32(1)
_cone_code(::Type{MOI.SecondOrderCone}) = Int32(2)
_cone_code(::Type{MOI.PositiveSemidefiniteConeTriangle}) = Int32(3)
_cone_code(::Type{MOI.ExponentialCone}) = Int32(4)
_cone_code(::Type{MOI.DualExponentialCone}) = Int32(5)
_cone_code(::Type{MOI.PowerCone{Float64}}) = Int32(6)
_cone_code(::Type{MOI.DualPowerCone{Float64}}) = Int32(7)
_cone_code(::Type{S}) where {S} = error("DiffOptB200.ConicModel: unsupported set $S")

"the per-cone parameter passed through conic_setup_ex: the exponent of a power cone, 0 for every other set"
_cone_param(set::Union{MOI.PowerCone{Float64},MOI.DualPowerCone{Float64}}) = set.exponent
_cone_param(::MOI.AbstractVectorSet) = 0.0

"cone list in row order (cone_type, cone_dim, cone_param) from the ProductOfSets -- what `Dπ` / `π` iterate over (diff_opt.jl:491-519)"
function _cone_list(model::ConicModel)
    entries = Tuple{Int,Int32,Int64,Float64}[]
    for (F, S) in MOI.get(model.model, MOI.ListOfConstraintTypesPresent())
        for ci in MOI.get(model.model, MOI.ListOfConstraintIndices{F,S}())
            r = MOI.Utilities.rows(model.model.constraints, ci)
            set = MOI.get(model.model, MOI.ConstraintSet(), ci)
            push!(entries, (first(r), _cone_code(S), Int64(length(r)), _cone_param(set)))
        end
    end
    sort!(entries; by = first)
    return Int32[e[2] for e in entries], Int64[e[3] for e in entries], Float64[e[4] for e in entries]
end

# _gradient_cache (ConicProgram.jl:172-255): A = -coefficients, b = constants, c (negated for MAX, zero for FEASIBILITY)
function _gradient_cache(model::ConicModel)
    model.cache_valid && return
    A = -convert(SparseArrays.SparseMatrixCSC{Float64,Int}, model.model.constraints.coefficients)
    b = model.model.constraints.constants
    if any(isnan, model.y) || length(model.y) < length(b)
        error("Some constraints are missing a value for the `ConstraintDualStart` attribute.")
    end
    if any(isnan, model.s) || length(model.s) < length(b)
        error("Some constraints are missing a value for the `ConstraintPrimalStart` attribute.")
    end
    n = size(A, 2)
    c = if MOI.get(model, MOI.ObjectiveSense()) == MOI.FEASIBILITY_SENSE
        zeros(n)
    else
        obj = MOI.get(model, MOI.ObjectiveFunction{MOI.ScalarAffineFunction{Float64}}())
        cc = Vector{Float64}(DiffOpt.sparse_array_representation(obj, n).terms)
        MOI.get(model, MOI.ObjectiveSense()) == MOI.MAX_SENSE ? -cc : cc
    end
    cone_type, cone_dim, cone_param = _cone_list(model)
    conic_setup(model.ctx, A, Vector{Float64}(b), c, model.x, model.s, model.y, cone_type, cone_dim, cone_param)
    model.vp = Vector{Float64}(undef, length(b))
    rc = ccall((:diffopt_b200_conic_get_vp, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int32), model.ctx.handle, model.vp, HOST)
    check(model.ctx, rc)
    model.cache_valid = true
    return
end

function DiffOpt.forward_differentiate!(model::ConicModel)
    model.diff_time = @elapsed begin
        _gradient_cache(model)
        m, n = size(model.model.constraints.coefficients)
        objective_function = DiffOpt._convert(MOI.ScalarAffineFunction{Float64}, model.input_cache.objective)
        dc = Vector{Float64}(DiffOpt.sparse_array_representation(objective_function, n).terms)
        db = zeros(m)
        DiffOpt._fill(S -> false, nothing, model.input_cache, model.model.constraints.sets, db)
        dAi = Int[]; dAj = Int[]; dAv = Float64[]
        DiffOpt._fill(S -> false, nothing, model.input_cache, model.model.constraints.sets, dAi, dAj, dAv)
        # (dA packed un-negated exactly as ConicProgram.jl:296-305 does; duplicates are summed on the device)
        r = conic_forward(model.ctx, n, m, Vector{Int64}(dAi), Vector{Int64}(dAj), dAv, db, dc;
                          atol = model.lsqr_atol, btol = model.lsqr_btol, conlim = model.lsqr_conlim)
        model.forw_grad_cache = CP.ForwCache(r.dz[1:n], r.dz[n+1:n+m], [r.dz[n+m+1]])
    end
    return nothing
end

function DiffOpt.reverse_differentiate!(model::ConicModel)
    model.diff_time = @elapsed begin
        _gradient_cache(model)
        m, n = size(model.model.constraints.coefficients)
        dx = zeros(n)
        for (vi, value) in model.input_cache.dx
            dx[vi.value] = value
        end
        r = conic_reverse(model.ctx, n, m, dx; atol = model.lsqr_atol, btol = model.lsqr_btol, conlim = model.lsqr_conlim)
        model.back_grad_cache = CP.ReverseCache(r.g, [model.x; model.vp; 1.0])
    end
    return nothing
end

# getters: same arithmetic as ConicProgram.jl:396-443 on the vectors that came back from the device
function MOI.get(model::ConicModel, ::DiffOpt.ReverseObjectiveFunction)
    g = model.back_grad_cache.g
    πz = model.back_grad_cache.πz
    dc = DiffOpt.lazy_combination(-, πz, g, length(g), eachindex(model.x))
    return DiffOpt.VectorScalarAffineFunction(dc, 0.0)
end

function MOI.get(model::ConicModel, ::DiffOpt.ForwardVariablePrimal, vi::MOI.VariableIndex)
    i = vi.value
    return -(model.forw_grad_cache.du[i] - model.x[i] * model.forw_grad_cache.dw[])
end

function DiffOpt._get_db(model::ConicModel, ci::MOI.ConstraintIndex{F,S}) where {F<:MOI.AbstractVectorFunction,S}
    i = MOI.Utilities.rows(model.model.constraints, ci)
    n = length(model.x)
    g = model.back_grad_cache.g
    πz = model.back_grad_cache.πz
    return DiffOpt.lazy_combination(-, πz, g, length(g), n .+ i)
end

function DiffOpt._get_dA(model::ConicModel, ci::MOI.ConstraintIndex{<:MOI.AbstractVectorFunction})
    i = MOI.Utilities.rows(model.model.constraints, ci)
    n = length(model.x)
    g = model.back_grad_cache.g
    πz = model.back_grad_cache.πz
    return g[n.+i] * πz[1:n]' - πz[n.+i] * g[1:n]'
end

# ------------------------------------------------------------------------------------------------
# (5) Batch-level entries used by training loops: shared weights, shared-parameter gradients, a lock-step batch of
#     conic problems, parameter pull-back (src/parameters.jl:341-534)
# ------------------------------------------------------------------------------------------------
const QP_SHARED_MATRICES = Int32(1)
const QP_SHARED_DIRECTION = Int32(2)
const QP_PACKED_Q = Int32(4)
const QP_ASYNC = Int32(8)
const QP_ALLREDUCE = Int32(16)

"reverse sensitivities of B problems that share Q, G, A (ONE instance each; an OptNet layer): `rev[n+m+p, B]`"
function qp_batch_reverse_shared(ctx::Context, Q::Matrix{Float64}, G::Matrix{Float64}, A::Matrix{Float64},
                                 h::Matrix{Float64}, z::Matrix{Float64}, lam::Matrix{Float64}, nu::Matrix{Float64},
                                 dl_dz::Matrix{Float64})
    n, B = size(z); m = size(G, 1); p = size(A, 1)
    rev = Matrix{Float64}(undef, n + m + p, B)
    info = zeros(Int32, B)
    rc = ccall((:diffopt_b200_qp_batch_solve_ex, LIB), Int32,
               (Ptr{Cvoid}, Int64, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Int32, Int32),
               ctx.handle, B, n, m, p, Q, G, A, h, z, lam, nu, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, dl_dz, C_NULL, rev,
               info, HOST, QP_SHARED_MATRICES)
    check(ctx, rc)
    return rev
end

"C layout of `diffopt_b200_coo_batch`: per-instance sparse triplets (0-based offsets `ptr`, Julia's 1-based `I`, `J`)"
struct CooBatch
    ptr::Ptr{Int64}
    I::Ptr{Int64}
    J::Ptr{Int64}
    V::Ptr{Float64}
end

"""
    qp_batch_forward_sparse(ctx, Q, G, A, h, z, lam, nu; dQ, dq, dG, dh, dA, db)

Forward sensitivities of B QPs whose direction matrices are the sparse triplets the reference itself builds: `dQ[b]`, `dG[b]`,
`dA[b]` are `SparseMatrixCSC` (QuadraticProgram.jl:396-424: `sparse(dGi, dGj, dGv, m, nv)` from the `_fill` of
src/diff_opt.jl:594-656) or `nothing`.  The right-hand side of :429-433 is assembled on the device; no dense direction exists.
"""
function qp_batch_forward_sparse(ctx::Context, Q::Array{Float64,3}, G::Array{Float64,3}, A::Array{Float64,3}, h::Matrix{Float64},
                                 z::Matrix{Float64}, lam::Matrix{Float64}, nu::Matrix{Float64};
                                 dQ = nothing, dq = nothing, dG = nothing, dh = nothing, dA = nothing, db = nothing)
    n, B = size(z); m = size(G, 1); p = size(A, 1)
    function triplets(mats)
        mats === nothing && return nothing
        ptr = zeros(Int64, B + 1); I = Int64[]; J = Int64[]; V = Float64[]
        for b in 1:B
            i, j, v = SparseArrays.findnz(mats[b])
            append!(I, i); append!(J, j); append!(V, v)
            ptr[b + 1] = length(V)
        end
        return (ptr, I, J, V)
    end
    tq, tg, ta = triplets(dQ), triplets(dG), triplets(dA)
    fwd = Matrix{Float64}(undef, n + m + p, B)
    info = zeros(Int32, B)
    ref(t) = t === nothing ? nothing : Ref(CooBatch(pointer(t[1]), pointer(t[2]), pointer(t[3]), pointer(t[4])))
    rq, rg, ra = ref(tq), ref(tg), ref(ta)
    cptr(r) = r === nothing ? Ptr{CooBatch}(C_NULL) : Base.unsafe_convert(Ptr{CooBatch}, r)
    vptr(v) = v === nothing ? Ptr{Float64}(C_NULL) : pointer(v)
    rc = GC.@preserve tq tg ta rq rg ra dq dh db ccall((:diffopt_b200_qp_batch_solve_coo, LIB), Int32,
               (Ptr{Cvoid}, Int64, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{CooBatch}, Ptr{Float64}, Ptr{CooBatch}, Ptr{Float64}, Ptr{CooBatch}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Int32, Int32),
               ctx.handle, B, n, m, p, Q, G, A, h, z, lam, nu, cptr(rq), vptr(dq), cptr(rg), vptr(dh), cptr(ra), vptr(db),
               C_NULL, fwd, C_NULL, info, HOST, Int32(0))
    check(ctx, rc)
    return fwd
end

"batch sum of the getters (QuadraticProgram.jl:307-314, :448-473) as one flat block [dQ | dq | dG | dh | dA | db]; `allreduce`: summed over the ranks of nccl_init"
function qp_batch_shared_grads(ctx::Context, z::Matrix{Float64}, lam::Matrix{Float64}, nu::Matrix{Float64}, rev::Matrix{Float64};
                               allreduce::Bool = false)
    n, B = size(z); m = size(lam, 1); p = size(nu, 1)
    out = Vector{Float64}(undef, n * n + n + m * n + m + p * n + p)
    rc = ccall((:diffopt_b200_qp_batch_shared_grads, LIB), Int32,
               (Ptr{Cvoid}, Int64, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Int32),
               ctx.handle, B, n, m, p, z, lam, nu, rev, out, HOST, allreduce ? QP_ALLREDUCE : Int32(0))
    check(ctx, rc)
    return out
end

"""
    param_pullback(ctx, term_param, term_index, term_coef, flat, nparams)

`reverse_differentiate!(::POI.Optimizer)` in array form (src/parameters.jl:341-534): `out[p] = sum coef * flat[index]` over the
parametric terms, `flat` the gradient block of `qp_batch_shared_grads`.  Index / coefficient of each term kind: see the header.
"""
function param_pullback(ctx::Context, term_param::Vector{Int64}, term_index::Vector{Int64}, term_coef::Vector{Float64},
                        flat::Vector{Float64}, nparams::Integer)
    out = Vector{Float64}(undef, nparams)
    rc = ccall((:diffopt_b200_param_pullback, LIB), Int32,
               (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Int32),
               ctx.handle, length(term_param), term_param, term_index, term_coef, length(flat), flat, nparams, out, HOST)
    check(ctx, rc)
    return out
end

"""
    conic_batch_reverse(ctx, problems, dx; atol, btol, conlim, maxiter)

`reverse_differentiate!` (ConicProgram.jl:336-394) of B conic problems of equal size in ONE persistent kernel.  `problems`:
vector of named tuples `(A, b, c, x, s, y, cone_type, cone_dim)` (and `cone_param` with power cones); `dx[n, B]`.  Returns `(g[n+m+1, B], dc[n, B], db[m, B], stats[4, B])`.
"""
function conic_batch_reverse(ctx::Context, problems::Vector, dx::Matrix{Float64};
                             atol = sqrt(eps()), btol = sqrt(eps()), conlim = 1 / sqrt(eps()), maxiter = 0)
    B = length(problems)
    rc = ccall((:diffopt_b200_conic_batch_begin, LIB), Int32, (Ptr{Cvoid}, Int64, Int32), ctx.handle, B, 1)
    check(ctx, rc)
    m, n = size(problems[1].A)
    for pr in problems
        A = pr.A::SparseArrays.SparseMatrixCSC{Float64,Int}
        cone_param = hasproperty(pr, :cone_param) ? Vector{Float64}(pr.cone_param) : zeros(length(pr.cone_type))
        rc = ccall((:diffopt_b200_conic_batch_add_ex, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                    Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Int32}, Ptr{Int64}, Ptr{Float64}, Int32),
                   ctx.handle, n, m, A.colptr, A.rowval, A.nzval, pr.b, pr.c, pr.x, pr.s, pr.y, length(pr.cone_type), pr.cone_type,
                   pr.cone_dim, cone_param, HOST)
        check(ctx, rc)
    end
    g = Matrix{Float64}(undef, n + m + 1, B); dc = Matrix{Float64}(undef, n, B); db = Matrix{Float64}(undef, m, B)
    stats = zeros(4, B)
    rc = ccall((:diffopt_b200_conic_batch_reverse, LIB), Int32,
               (Ptr{Cvoid}, Ptr{Float64}, Float64, Float64, Float64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32),
               ctx.handle, dx, atol, btol, conlim, maxiter, g, dc, db, stats, HOST)
    check(ctx, rc)
    return (g = g, dc = dc, db = db, stats = stats)
end

# ------------------------------------------------------------------------------------------------
# (6) NonLinearProgram backend: the factorisation hook `model.input_cache.factorization(M, model)`
#     (nlp_utilities.jl:436-444; default `_lu_with_inertia_correction`, NonLinearProgram.jl:402-435).  The returned object
#     only has to support `ldiv!(ds, K, N)`; `nothing` means the correction failed.
#     usage:  MOI.set(model, DiffOpt.NonLinearKKTJacobianFactorization(), DiffOptB200.nlp_factorization(ctx))
# ------------------------------------------------------------------------------------------------
struct InertiaCorrectedLU
    ctx::Context
    N::Int
    corrections::Int
end

function nlp_factorization(ctx::Context; st = 1e-6, max_corrections = 50)
    return function (M::SparseArrays.SparseMatrixCSC{Float64,Int}, model)
        NLP = DiffOpt.NonLinearProgram
        num_w = NLP._get_num_primal_vars(model) + length(model.cache.leq_locations) + length(model.cache.geq_locations)
        num_cons = NLP._get_num_constraints(model)
        nc = Ref{Int32}(0)
        rc = ccall((:diffopt_b200_sparse_setup_inertia, LIB), Int32,
                   (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64, Int64, Float64, Int32, Ptr{Int32}),
                   ctx.handle, size(M, 1), M.colptr, M.rowval, M.nzval, num_w, num_cons, st, max_corrections, nc)
        rc < 0 && check(ctx, rc)
        if rc > 0
            @warn "Inertia correction failed."
            return nothing
        end
        return InertiaCorrectedLU(ctx, size(M, 1), Int(nc[]))
    end
end

function LinearAlgebra.ldiv!(ds::Matrix{Float64}, K::InertiaCorrectedLU, N::AbstractMatrix)
    Nd = Matrix{Float64}(N)
    rc = ccall((:diffopt_b200_sparse_solve, LIB), Int32, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Int32),
               K.ctx.handle, size(Nd, 2), Nd, ds, HOST)
    check(K.ctx, rc)
    return ds
end

end # module
