# ConicIPB200.jl -- the Julia-side binding a ConicIP.jl maintainer adds to use the B200 engine.
#
# It is a thin `ccall` shim over libconicip_b200.so (include/conicip_b200.h): no CUDA.jl, no kernel
# generation, no CPU fallback.  `kktsolver_b200` has exactly the signature of
# `ConicIP.kktsolver_qr` / `pivot(ConicIP.kktsolver_2x2)` (src/kktsolvers.jl:18,349), so
#
#     sol = conicIP(Q, c, A, b, cone_dims, G, d; kktsolver = ConicIPB200.kktsolver_b200)
#
# is the whole integration.  Julia is not installed in the build image, so this file is not
# executed by the test-suite; tests/ drive the same C symbols through ctypes (_lib.py) with the
# identical call sequence.
module ConicIPB200

using LinearAlgebra, SparseArrays
import ConicIP
using ConicIP: Block, VecCongurance
using ConicIP.WoodburyMatrices: SymWoodbury

const LIB = get(ENV, "CONICIP_B200_LIB", joinpath(@__DIR__, "..", "libconicip_b200.so"))

const CONE_CODE = Dict("R" => Cint(0), "Q" => Cint(1), "S" => Cint(2))
const BLK_DIAG, BLK_WOODBURY, BLK_VECCONG = Cint(0), Cint(1), Cint(2)

struct Options            # mirrors cip_options
    struct_size::Cint
    device::Cint
    reg_delta::Cdouble
    reg_eps_G::Cdouble
    q_kind::Cint
    verbose::Cint
    dist_chol::Cint
    aug_rho::Cdouble
    ngpus::Cint           # > 1: this one process drives that many GPUs behind the handle (rows of A sliced on cone boundaries)
    fold_scaling::Cint    # 0 auto, 1 always, 2 never: R-only problems without a second (scaled) copy of A
    row_structure::Cint   # 1: singleton R rows go onto the diagonal of H, the SYRK runs on the other rows (one GPU);
                          # 2: also factor H as its diagonal plus the coupled block H_KK (no n x n buffer)
end
make_options(; device = -1, reg_delta = 0.0, q_kind = 0, ngpus = 1, fold_scaling = 0, row_structure = 0) =
    Options(Cint(sizeof(Options)), Cint(device), reg_delta, 0.0, Cint(q_kind), Cint(0), Cint(-1), -1.0, Cint(ngpus),
            Cint(fold_scaling), Cint(row_structure))

lasterr() = unsafe_string(ccall((:cip_last_error, LIB), Cstring, ()))
function check(rc::Cint)
    rc < 0 && error("conicip_b200: ", lasterr())
    return rc
end

struct Csc                # mirrors cip_csc: a SparseMatrixCSC{Float64,Int64} passed field by field
    nrows::Cint
    ncols::Cint
    colptr::Ptr{Int64}
    rowval::Ptr{Int64}
    nzval::Ptr{Cdouble}
    index_base::Cint
end
Csc(M::SparseMatrixCSC{Float64,Int64}) = Csc(size(M, 1), size(M, 2), pointer(M.colptr), pointer(M.rowval), pointer(M.nzval), 1)

mutable struct Engine
    h::Ptr{Cvoid}
    n::Int; m::Int; p::Int
    function Engine(Q, A, G, cone_dims; reg_delta = 0.0, ngpus = 1, device = -1, fold_scaling = 0, row_structure = 0)
        n = size(Q, 1); m = size(A, 1); p = size(G, 1)
        if A isa SparseMatrixCSC          # sparse LEVEL 1: no dense copy on the host (cip_create_csc)
            Qs = SparseMatrixCSC{Float64,Int64}(sparse(Q)); As = SparseMatrixCSC{Float64,Int64}(A)
            Gs = SparseMatrixCSC{Float64,Int64}(sparse(G))
            ct = Cint[CONE_CODE[t] for (t, _) in cone_dims]; cdim = Cint[k for (_, k) in cone_dims]
            opts = Ref(make_options(; device, reg_delta, q_kind = 2, ngpus, fold_scaling, row_structure))
            hp = Ref{Ptr{Cvoid}}(C_NULL)
            GC.@preserve Qs As Gs begin
                rc = ccall((:cip_create_csc, LIB), Cint,
                           (Ref{Ptr{Cvoid}}, Cint, Ref{Csc}, Ref{Csc}, Ref{Csc}, Cint, Ptr{Cint}, Ptr{Cint}, Ref{Options}),
                           hp, n, Ref(Csc(Qs)), Ref(Csc(As)), Ref(Csc(Gs)), length(ct), ct, cdim, opts)
            end
            rc != 0 && error("cip_create_csc: ", lasterr())
            e = new(hp[], n, m, p)
            finalizer(x -> ccall((:cip_destroy, LIB), Cint, (Ptr{Cvoid},), x.h), e)
            return e
        end
        # Julia arrays are column-major: dense copies are passed as they are (SURVEY 8b "Argument types")
        Qd = Q isa Diagonal ? collect(Q.diag) : Matrix{Float64}(Q)
        qk = Q isa Diagonal ? Cint(1) : Cint(0)
        Ad = Matrix{Float64}(A)
        Gd = Matrix{Float64}(G)
        ct = Cint[CONE_CODE[t] for (t, _) in cone_dims]
        cdim = Cint[k for (_, k) in cone_dims]
        opts = Ref(make_options(; device, reg_delta, q_kind = qk, ngpus, fold_scaling, row_structure))
        hp = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:cip_create, LIB), Cint,
                   (Ref{Ptr{Cvoid}}, Cint, Cint, Cint, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Cint,
                    Ptr{Cdouble}, Cint, Cint, Ptr{Cint}, Ptr{Cint}, Ref{Options}),
                   hp, n, m, p, Qd, max(n, 1), Ad, max(m, 1), Gd, max(p, 1),
                   length(ct), ct, cdim, opts)
        rc != 0 && error("cip_create: ", lasterr())
        e = new(hp[], n, m, p)
        finalizer(x -> ccall((:cip_destroy, LIB), Cint, (Ptr{Cvoid},), x.h), e)   # handle lifetime = closure lifetime
        return e
    end
end

# Flatten a ConicIP `Block` (src/blockmatrices.jl:35-43) into the arrays of cip_factor.
# The first call of a solve passes Diagonal(ones) for every cone, Q/S slots included
# (src/ConicIP.jl:704) -- the per-call `kind` array covers that.
function flatten(F::Block)
    nc = length(F.Blocks)
    kind = Vector{Cint}(undef, nc); fD = zeros(nc)
    fa = Float64[]; fb = Float64[]; fR = Float64[]
    for (i, B) in enumerate(F.Blocks)
        if B isa Diagonal
            kind[i] = BLK_DIAG; append!(fa, B.diag); append!(fb, zeros(length(B.diag)))
        elseif B isa SymWoodbury
            # only the rank-1 form nestod_soc builds (src/ConicIP.jl:192) has a flat representation; the general
            # WoodburyMatrices form (matrix B, matrix D: src/blockmatrices.jl:135-141) is rejected, not mangled
            (size(B.B, 2) == 1 && length(B.D) == 1) ||
                error("ConicIPB200: SymWoodbury blocks of rank > 1 are not supported (block $i has rank $(size(B.B, 2)))")
            kind[i] = BLK_WOODBURY
            append!(fa, B.A.diag); append!(fb, vec(B.B)); fD[i] = B.D isa Number ? B.D : B.D[1, 1]
        elseif B isa VecCongurance
            kind[i] = BLK_VECCONG
            k = size(B, 1); append!(fa, zeros(k)); append!(fb, zeros(k)); append!(fR, vec(B.R))
        else
            error("unsupported scaling block type $(typeof(B))")
        end
    end
    return kind, fa, fb, fD, fR
end

"""
    kktsolver_b200(Q, A, G, cone_dims) -> solve3x3gen

Drop-in for `kktsolver_qr` / `pivot(kktsolver_2x2)`; three-level closure protocol of
docs/src/guides/kkt_solvers.md:84-109.
"""
function kktsolver_b200(Q, A, G, cone_dims; engine_options...)
    eng = Engine(Q, A, G, cone_dims; engine_options...)               # LEVEL 1: upload once

    function solve3x3gen(F, F⁻ᵀ)                                      # LEVEL 2: form H, factor
        kind, fa, fb, fD, fR = flatten(F)
        rc = ccall((:cip_factor, LIB), Cint,
                   (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}),
                   eng.h, kind, fa, fb, fD, isempty(fR) ? C_NULL : pointer(fR))
        check(rc)                 # rc > 0: non-PD pivot -> NaN results -> status :Error (src/ConicIP.jl:870-873)
        failed = rc > 0

        function solve3x3(y, w, v)                                    # LEVEL 3: solve
            a = Vector{Float64}(undef, eng.n)                         # fresh outputs (mutated by axpy4!, :920)
            b = Vector{Float64}(undef, eng.p)
            c = Vector{Float64}(undef, eng.m)
            if failed
                fill!(a, NaN); fill!(b, NaN); fill!(c, NaN)
                return (a, b, c)
            end
            check(ccall((:cip_solve, LIB), Cint,
                        (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}),
                        eng.h, Vector{Float64}(y), Vector{Float64}(w), Vector{Float64}(v), a, b, c))
            return (a, b, c)
        end
        return solve3x3
    end
    return solve3x3gen
end

"""
    solve_multi(eng, Y, W, V) -> (A, B, C)

Several right-hand sides (the columns of `Y` n x k, `W` p x k, `V` m x k) through the current factorisation of
`eng` in one `ccall` (`cip_solve_multi`): the two products with `A` are shared by pairs of columns.  `conicIP`
itself cannot use it (its corrector right-hand side depends on the predictor's solution, src/ConicIP.jl:879-907);
it is for callers with independent right-hand sides.
"""
function solve_multi(eng, Y::Matrix{Float64}, W::Matrix{Float64}, V::Matrix{Float64})
    k = size(Y, 2)
    A = Matrix{Float64}(undef, eng.n, k); B = Matrix{Float64}(undef, eng.p, k); C = Matrix{Float64}(undef, eng.m, k)
    check(ccall((:cip_solve_multi, LIB), Cint,
                (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}),
                eng.h, k, Y, eng.n, W, max(eng.p, 1), V, eng.m, A, B, C))
    return (A, B, C)
end

struct StructureInfo      # mirrors cip_structure_t
    struct_size::Cint
    enabled::Cint
    singleton_rows::Cint
    empty_rows::Cint
    rest_rows::Cint
    rest_cols::Cint
    compressed::Cint
    base_has_gtg::Cint
end
"""
    structure_info(eng) -> StructureInfo

How an engine created with `row_structure = 1` split the rows of `A` (`cip_structure_info`).
"""
function structure_info(eng::Engine)
    r = Ref(StructureInfo(Cint(sizeof(StructureInfo)), 0, 0, 0, 0, 0, 0, 0))
    check(ccall((:cip_structure_info, LIB), Cint, (Ptr{Cvoid}, Ref{StructureInfo}), eng.h, r))
    return r[]
end
struct SplitInfo          # mirrors cip_split_t
    struct_size::Cint
    enabled::Cint
    coupled_cols::Cint
    diagonal_cols::Cint
    cols_from_rest::Cint
    cols_from_Q::Cint
    cols_from_G::Cint
end
"""
    split_info(eng) -> SplitInfo

How an engine created with `row_structure = 2` split the columns of `H` (`cip_split_info`): `coupled_cols` columns
form the dense block `H_KK`, `diagonal_cols` hold only their diagonal.  `cols_from_rest`, `cols_from_Q` and
`cols_from_G` count why a column is coupled (a rest row of `A`, an off-diagonal entry of `Q`, `G` when
`aug_rho > 0`); the sets overlap.  All zero for other engines.
"""
function split_info(eng::Engine)
    r = Ref(SplitInfo(Cint(sizeof(SplitInfo)), 0, 0, 0, 0, 0, 0))
    check(ccall((:cip_split_info, LIB), Cint, (Ptr{Cvoid}, Ref{SplitInfo}), eng.h, r))
    return r[]
end
"""
    kktsolver_b200(; ngpus = 8, ...) -> kktsolver

Options bound: `conicIP(Q, c, A, b, cone_dims, G, d; kktsolver = kktsolver_b200(ngpus = 8))` row-shards `A` over
eight GPUs of this process behind the one callback the reference makes (src/ConicIP.jl:667).
"""
kktsolver_b200(; engine_options...) = (Q, A, G, cone_dims) -> kktsolver_b200(Q, A, G, cone_dims; engine_options...)

# ---- cone kernels (no callback exists for these in conicIP; a device-resident driver calls them)
nt_scaling!(eng::Engine, v, s, λ) = check(ccall((:cip_nt_scaling, LIB), Cint,
    (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), eng.h, v, s, λ))
function maxstep(eng::Engine, x, d = nothing; scale = 1.0)
    α = Ref{Cdouble}(0.0)
    check(ccall((:cip_maxstep, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Cdouble, Ref{Cdouble}),
                eng.h, x, d === nothing ? C_NULL : pointer(d), scale, α))
    return α[]
end
apply!(eng::Engine, op::Integer, x, y) = check(ccall((:cip_apply, LIB), Cint,
    (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Ptr{Cdouble}), eng.h, op, x, y))
cone_prod!(eng::Engine, o, x, y) = check(ccall((:cip_cone_prod, LIB), Cint,
    (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), eng.h, x, y, o))
cone_div!(eng::Engine, o, x, y) = check(ccall((:cip_cone_div, LIB), Cint,
    (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), eng.h, x, y, o))

# ---- the whole solve behind one ccall (cip_ipm_solve; SURVEY 8f rank 1): same arguments, options
# and `Solution` as `ConicIP.conicIP`, with the loop of src/ConicIP.jl:468-939 running in the library
# on device-resident vectors.
struct IpmOptions
    struct_size::Cint; maxIters::Cint; maxRefinementSteps::Cint; verbose::Cint
    optTol::Cdouble; DTB::Cdouble; infeasTol::Cdouble; refinementThreshold::Cdouble
end
struct IpmResult
    status::Cint; Iter::Cint; factors::Cint; solves::Cint
    Mu::Cdouble; prFeas::Cdouble; duFeas::Cdouble; muFeas::Cdouble; pobj::Cdouble; dobj::Cdouble; seconds::Cdouble
end
const STATUS = (:None, :Optimal, :Infeasible, :Unbounded, :Abandoned, :Error)

function conicIP_b200(Q, c::AbstractVector, A, b::AbstractVector, cone_dims,
                      G = spzeros(0, length(c)), d = zeros(0);
                      optTol = 1e-6, DTB = 0.01, verbose = false, maxRefinementSteps = 3, maxIters = 100,
                      infeasTol = optTol, refinementThreshold = optTol / 1e7, ngpus = 1, device = -1)
    eng = Engine(Q, A, G, cone_dims; ngpus, device)
    y = Vector{Float64}(undef, eng.n); w = Vector{Float64}(undef, eng.p); v = Vector{Float64}(undef, eng.m)
    opts = Ref(IpmOptions(Cint(sizeof(IpmOptions)), maxIters, maxRefinementSteps, verbose, optTol, DTB, infeasTol,
                          refinementThreshold))
    res = Ref(IpmResult(0, 0, 0, 0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0))
    check(ccall((:cip_ipm_solve, LIB), Cint,
                (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{IpmOptions}, Ptr{Cdouble}, Ptr{Cdouble},
                 Ptr{Cdouble}, Ref{IpmResult}),
                eng.h, Vector{Float64}(c), Vector{Float64}(b), Vector{Float64}(d), opts, y, w, v, res))
    r = res[]
    return ConicIP.Solution(y, w, v, STATUS[r.status + 1], r.Iter, r.Mu, r.prFeas, r.duFeas, r.muFeas, r.pobj, r.dobj)
end

# ---- preprocessor (SURVEY 8f rank 4): drop-in for ConicIP.imcols (src/preprocessor.jl:10-28) on the device.
# Returns (R, consistent) with 1-based sorted row indices, R empty when the system is inconsistent.
function imcols_b200(A, b, ϵ = 1e-8; device = -1)
    Ad = Matrix{Float64}(A); p, n = size(Ad)
    keep = zeros(Cint, max(p, 1)); nkeep = Ref{Cint}(0); cons = Ref{Cint}(1)
    check(ccall((:cip_imcols, LIB), Cint,
                (Cint, Ptr{Cdouble}, Cint, Cint, Cint, Ptr{Cdouble}, Cdouble, Ptr{Cint}, Ref{Cint}, Ref{Cint}),
                device, Ad, max(p, 1), p, n, Vector{Float64}(b), ϵ, keep, nkeep, cons))
    cons[] == 0 && return (Int[], false)
    return (findall(!iszero, keep[1:p]), true)
end
# `preprocess_conicIP` itself needs no change beyond calling imcols_b200 at src/preprocessor.jl:58-59.

# ---- MOI / JuMP (SURVEY 8f rank 2).  `ConicIP.Optimizer` has no kktsolver field (src/MOI_wrapper.jl:19-31) and
# `optimize!` forwards only verbose / optTol / maxIters to `preprocess_conicIP` (:278-282), which itself forwards any
# extra option to `conicIP` (src/preprocessor.jl:44,82-84).  Two ways to select the engine from JuMP:
#
#  (1) the two-line patch `julia/MOI_wrapper_kktsolver.patch` (one struct field, one keyword), after which
#          model = Model(() -> ConicIP.Optimizer(kktsolver = ConicIPB200.kktsolver_b200(ngpus = 8)))
#
#  (2) without touching ConicIP.jl: `ConicIPB200.Optimizer`, a wrapper optimizer that owns a stock
#      `ConicIP.Optimizer`, delegates the whole MOI interface to it, and for the solve itself re-runs the stock
#      `optimize!` with `ConicIP.preprocess_conicIP` intercepted so that `kktsolver =` is added to its options.
import MathOptInterface
const MOI = MathOptInterface

"""
    ConicIPB200.Optimizer(; ngpus = 1, verbose = false, optTol = 1e-6, maxIters = 100)

Drop-in for `ConicIP.Optimizer` (src/MOI_wrapper.jl:19-40) whose KKT systems are solved by the B200 engine.
"""
mutable struct Optimizer <: MOI.AbstractOptimizer
    inner::ConicIP.Optimizer
    kktsolver::Function
end
Optimizer(; ngpus = 1, device = -1, kwargs...) = Optimizer(ConicIP.Optimizer(; kwargs...), kktsolver_b200(; ngpus, device))

# the model data path of the stock optimizer is re-used as it is (constraint extraction :102-136, :185-275)
for f in (:empty!, :is_empty)
    @eval MOI.$f(o::Optimizer) = MOI.$f(o.inner)
end
MOI.get(::Optimizer, ::MOI.SolverName) = "ConicIP (B200 KKT engine)"
MOI.get(o::Optimizer, attr::MOI.AnyAttribute, args...) = MOI.get(o.inner, attr, args...)
MOI.supports(o::Optimizer, attr::MOI.AnyAttribute, args...) = MOI.supports(o.inner, attr, args...)
MOI.supports_constraint(o::Optimizer, F::Type{<:MOI.AbstractFunction}, S::Type{<:MOI.AbstractSet}) =
    MOI.supports_constraint(o.inner, F, S)
MOI.set(o::Optimizer, attr::MOI.AnyAttribute, args...) = MOI.set(o.inner, attr, args...)

# `optimize!(dest, src)` (src/MOI_wrapper.jl:142-285) builds Q, c, A, b, cone_dims, G, d and calls
# `preprocess_conicIP(...; verbose, optTol, maxIters)` at :278.  The solve is re-issued through the same function
# with the engine's kktsolver appended to the options, by shadowing the name in a module that `include`s the
# stock wrapper code path unchanged:
function MOI.optimize!(dest::Optimizer, src::MOI.ModelLike)
    return with_kktsolver(dest.kktsolver) do
        MOI.optimize!(dest.inner, src)
    end
end
# task-local override consulted by the patched-in keyword default below
const KKTSOLVER_OVERRIDE = Ref{Union{Nothing,Function}}(nothing)
function with_kktsolver(f, k::Function)
    old = KKTSOLVER_OVERRIDE[]
    KKTSOLVER_OVERRIDE[] = k
    try
        return f()
    finally
        KKTSOLVER_OVERRIDE[] = old
    end
end
# `conicIP`'s keyword default is `kktsolver = kktsolver_qr` (src/ConicIP.jl:498); the reference exports that
# function, so a method on it that consults the override routes every stock call site -- including the one
# `optimize!` reaches through `preprocess_conicIP` -- to the engine while a `ConicIPB200.Optimizer` is solving,
# and falls back to the stock QR solver otherwise.
# The stock method is reached through the world age recorded just before the route is installed
# (`Base.invoke_in_world`): binding `ConicIP.kktsolver_qr` to a constant would not do, because redefining the
# method changes what that very function object calls.
const STOCK_WORLD = Ref{UInt}(typemax(UInt))
function routed_kktsolver(Q, A, G, cone_dims)
    k = KKTSOLVER_OVERRIDE[]
    k === nothing || return k(Q, A, G, cone_dims)
    return Base.invoke_in_world(STOCK_WORLD[], ConicIP.kktsolver_qr, Q, A, G, cone_dims)
end
# Installing the route is one method definition in ConicIP's namespace (done once, at `using ConicIPB200`); with the
# patch of (1) applied it is unnecessary and skipped.
function __init__()
    if !(:kktsolver in fieldnames(ConicIP.Optimizer))
        STOCK_WORLD[] = Base.get_world_counter()
        @eval ConicIP kktsolver_qr(Q, A, G, cone_dims) = $(routed_kktsolver)(Q, A, G, cone_dims)
    end
end

end # module
