# B200KKT.jl -- the shim a MadNLP.jl maintainer adds to drive libb200kkt.so (include/b200kkt.h) from MadNLP's
# existing plugin surface.  NOT RUN in this repository's CI (no Julia in the build image); it is the reference-side
# binding INTEGRATION.md describes, kept next to the library so that the C ABI and its consumer evolve together.
#
#   using MadNLP, MadNLPGPU, CUDA
#   include("B200KKT.jl"); using .B200KKT
#   madnlp(nlp; kkt_system = MadNLP.SparseCondensedKKTSystem, linear_solver = B200KKT.B200Solver,
#          equality_treatment = MadNLP.RelaxEquality, tol = 1e-4)
#
# Interface implemented (src/LinearSolvers/linearsolvers.jl:13-95; same list every plugin imports,
# lib/MadNLPHSL/src/MadNLPHSL.jl:3-32): constructor(csc; opt, logger), factorize!, solve_linear_system!, is_inertia,
# inertia, improve!, introduce, input_type, default_options, is_supported, is_async.
module B200KKT

import MadNLP
import MadNLP: AbstractLinearSolver, AbstractOptions, MadNLPLogger, SymbolicException, FactorizationException,
    SolveException, factorize!, solve_linear_system!, is_inertia, inertia, improve!, introduce, input_type,
    default_options, is_supported, is_async
using CUDA, CUDA.CUSPARSE
# (nothing here extends a method on types this module does not own without one of ITS types in the signature)

const libb200kkt = get(ENV, "B200KKT_LIB", "libb200kkt.so")

# mirror of `struct b2_options` (include/b200kkt.h)
Base.@kwdef mutable struct B200Options <: AbstractOptions
    b200_ordering::Int32 = 0            # B2_ORDER_METIS_ND
    b200_nemin::Int32 = 16
    b200_relax_zeros::Float64 = 0.25
    b200_pivot_eps::Float64 = 1e-13
    b200_use_cuda_graph::Int32 = 1
    b200_small_front_max::Int32 = 160
    b200_kkt_n_primal::Int32 = 0        # set by the KKT overloads below for SparseKKTSystem
    b200_fuse_max_fronts::Int32 = 8
    b200_dep_schedule::Int32 = 1
    b200_chain_merge_f::Int32 = 0
    # B200DenseSolver only: MadNLP.BUNCHKAUFMAN (what LapackCPUSolver / LapackCUDASolver default to) selects Bunch-Kaufman
    # pivoting (B2_PIVOT_BUNCH_KAUFMAN); `nothing` keeps the static 1 x 1 pivots.  The sparse solver always pivots statically.
    lapack_algorithm::Union{Nothing,MadNLP.LinearFactorization} = nothing
end

struct CB2Options
    ordering::Int32; nemin::Int32; relax_zeros::Float64; pivot_eps::Float64
    use_cuda_graph::Int32; small_front_max::Int32; n_parts::Int32; part_rank::Int32
    kkt_n_primal::Int32; fuse_max_fronts::Int32; dep_schedule::Int32; chain_merge_f::Int32
    pivoting::Int32; reserved::NTuple{3,Int32}
end
CB2Options(o::B200Options; dense::Bool = false) = CB2Options(o.b200_ordering, o.b200_nemin, o.b200_relax_zeros, o.b200_pivot_eps,
    o.b200_use_cuda_graph, o.b200_small_front_max, 1, 0, o.b200_kkt_n_primal, o.b200_fuse_max_fronts, o.b200_dep_schedule, o.b200_chain_merge_f,
    Int32(dense && o.lapack_algorithm == MadNLP.BUNCHKAUFMAN ? 1 : 0), ntuple(_ -> Int32(0), 3))

last_error() = unsafe_string(ccall((:b2_last_error, libb200kkt), Cstring, ()))
function check(rc::Cint, exc)
    rc == 0 && return
    rc == 3 && throw(SymbolicException())
    rc == 4 && throw(FactorizationException())
    rc == 5 && throw(SolveException())
    error("b200kkt error $rc: $(last_error())")
end

mutable struct B200Solver{T} <: AbstractLinearSolver{T}
    handle::Ptr{Cvoid}
    tril::CuSparseMatrixCSC{T,Int32}    # kept by reference: values are re-read on every factorize! (cudss.jl:154-158)
    opt::B200Options
    logger::MadNLPLogger
end

function B200Solver(csc::CuSparseMatrixCSC{Float64,Int32}; opt = B200Options(), logger = MadNLPLogger())
    n = size(csc, 1)
    colptr = Array(csc.colPtr) .- Int32(1)          # host, 0-based (analysis runs on the host, once)
    rowval = Array(csc.rowVal) .- Int32(1)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    copt = Ref(CB2Options(opt))
    rc = ccall((:b2_create, libb200kkt), Cint,
        (Int32, Int64, Ptr{Int32}, Ptr{Int32}, CuPtr{Float64}, Ptr{CB2Options}, Ptr{Int32}, Ptr{Ptr{Cvoid}}),
        n, length(rowval), colptr, rowval, pointer(csc.nzVal), copt, C_NULL, h)
    check(rc, SymbolicException)
    M = B200Solver{Float64}(h[], csc, opt, logger)
    finalizer(m -> ccall((:b2_destroy, libb200kkt), Cint, (Ptr{Cvoid},), m.handle), M)
    return M
end

stream_ptr() = Ptr{Cvoid}(UInt(CUDA.stream().handle))

function factorize!(M::B200Solver)
    check(ccall((:b2_factorize, libb200kkt), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), M.handle, stream_ptr()), FactorizationException)
    return M
end

function solve_linear_system!(M::B200Solver{T}, x::CuVector{T}) where T
    check(ccall((:b2_solve, libb200kkt), Cint, (Ptr{Cvoid}, CuPtr{T}, Int32, Ptr{Cvoid}), M.handle, pointer(x), 1, stream_ptr()), SolveException)
    return x
end

is_inertia(::B200Solver) = true
function inertia(M::B200Solver)
    p = Ref{Int64}(0); z = Ref{Int64}(0); n = Ref{Int64}(0)
    check(ccall((:b2_inertia, libb200kkt), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Cvoid}),
        M.handle, p, z, n, stream_ptr()), FactorizationException)
    return (Int(p[]), Int(z[]), Int(n[]))       # (num_pos, num_zero, num_neg): the order src/IPM/solver.jl:626 destructures
end

function improve!(M::B200Solver)
    ch = Ref{Int32}(0)
    ccall((:b2_improve, libb200kkt), Cint, (Ptr{Cvoid}, Ptr{Int32}), M.handle, ch)
    return ch[] != 0
end

introduce(::B200Solver) = "b200kkt (sm_100a multifrontal LDL')"
input_type(::Type{<:B200Solver}) = :csc
default_options(::Type{<:B200Solver}) = B200Options()
is_supported(::Type{<:B200Solver}, ::Type{Float64}) = true
is_supported(::Type{<:B200Solver}, ::Type{Float32}) = false
is_async(::B200Solver) = true

# ---------------------------------------------------------------------------------------------------------------------
# KKT-level overloads.  Dispatch is on OUR solver type in the `LS` parameter of the stock KKT structs
#   SparseCondensedKKTSystem{T,VT,MT,QN,LS,...} (src/KKT/Sparse/condensed.jl:7)   with VT <: CuVector AND LS <: B200Solver
#   DenseCondensedKKTSystem{T,VT,MT,QN,LS,VI}   (src/KKT/Dense/condensed.jl:10)   with VT <: CuVector AND LS <: B200DenseSolver
# -- strictly more specific than MadNLPGPU's `VT <: AbstractGPUVector` methods (lib/MadNLPGPU/src/KKT/gpu_sparse.jl:308-382,
# gpu_dense.jl:86-138), so loading both packages is neither ambiguous nor type piracy (a type this module owns is in every
# signature).  The native plans live in the solver object (which this module owns), built lazily from the kkt's own maps at
# the first call: MadNLP's `ext` slot (get_sparse_condensed_ext, gpu_sparse.jl:100-130) keeps whatever MadNLPGPU put there.
# ---------------------------------------------------------------------------------------------------------------------
mutable struct CondensedPlans
    cond::Ptr{Cvoid}        # b2_condensed_plan   (pattern of tril(H) U diag U tril(Jt Jt') + the dptr/hptr/jptr maps)
    hess_plan::Ptr{Cvoid}   # b2_transfer_plan    hess_raw (COO) -> hess_com (CSC)
    jt_plan::Ptr{Cvoid}     # b2_transfer_plan    jt_coo         -> jt_csc
    hess_spmv::Ptr{Cvoid}   # b2_spmv_plan of hess_com
    jt_spmv::Ptr{Cvoid}     # b2_spmv_plan of jt_csc
    bounds::Ptr{Cvoid}      # b2_bounds (ind_lb / ind_ub and their inverse maps)
end

const _plans = IdDict{Any,CondensedPlans}()     # solver handle -> plans (freed with the solver)

const B200CondensedKKT{T} = MadNLP.SparseCondensedKKTSystem{T,VT,MT,QN,LS} where {VT<:CuVector{T},MT,QN,LS<:B200Solver}

function plans(kkt::B200CondensedKKT{T}) where T
    get!(_plans, kkt.linear_solver) do
        n = size(kkt.hess_com, 1); m = size(kkt.jt_csc, 2)
        h0(v) = Array(v) .- one(eltype(v))                                   # host, 0-based
        hcp, hrv = h0(kkt.hess_com.colPtr), h0(kkt.hess_com.rowVal)
        jcp, jrv = h0(kkt.jt_csc.colPtr), h0(kkt.jt_csc.rowVal)
        cond = Ref{Ptr{Cvoid}}(C_NULL); nnz_aug = Ref{Int64}(0)
        check(ccall((:b2_condensed_symbolic, libb200kkt), Cint,
            (Int32, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Ptr{Cvoid}}, Ptr{Int64}),
            n, m, hcp, hrv, jcp, jrv, cond, nnz_aug), SymbolicException)
        @assert nnz_aug[] == length(MadNLP.nzval(kkt.aug_com))               # same pattern as build_condensed_aug_symbolic
        tplan(map_d) = begin
            mp = Array(map_d) .- 1; h = Ref{Ptr{Cvoid}}(C_NULL)
            check(ccall((:b2_transfer_plan_create, libb200kkt), Cint, (Int64, Int64, Ptr{Int64}, Ptr{Ptr{Cvoid}}),
                length(mp), maximum(mp; init = -1) + 1, mp, h), SymbolicException); h[]
        end
        splan(nr, nc, cp, rv) = begin
            h = Ref{Ptr{Cvoid}}(C_NULL)
            check(ccall((:b2_spmv_plan_create, libb200kkt), Cint, (Int32, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Ptr{Cvoid}}), nr, nc, cp, rv, h), SymbolicException); h[]
        end
        lb = Array(kkt.ind_lb) .- 1; ub = Array(kkt.ind_ub) .- 1; b = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:b2_bounds_create, libb200kkt), Cint, (Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Ptr{Cvoid}}),
            length(kkt.pr_diag), length(lb), length(ub), lb, ub, b), SymbolicException)
        CondensedPlans(cond[], tplan(kkt.hess_csc_map), tplan(kkt.jt_csc_map), splan(n, n, hcp, hrv), splan(n, m, jcp, jrv), b[])
    end
end

function MadNLP.build_kkt!(kkt::B200CondensedKKT{T}) where T
    p = plans(kkt)
    check(ccall((:b2_condensed_assemble, libb200kkt), Cint,
        (Ptr{Cvoid}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        p.cond, pointer(MadNLP.nzval(kkt.aug_com)), pointer(kkt.pr_diag), pointer(kkt.du_diag),
        pointer(MadNLP.nzval(kkt.hess_com)), pointer(MadNLP.nzval(kkt.jt_csc)), pointer(kkt.diag_buffer), stream_ptr()), FactorizationException)
end

function MadNLP.compress_hessian!(kkt::B200CondensedKKT{T}) where T
    check(ccall((:b2_transfer, libb200kkt), Cint, (Ptr{Cvoid}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        plans(kkt).hess_plan, pointer(MadNLP.nzval(kkt.hess_com)), pointer(kkt.hess_raw.V), stream_ptr()), FactorizationException)
end

function MadNLP.compress_jacobian!(kkt::B200CondensedKKT{T}) where T
    check(ccall((:b2_transfer, libb200kkt), Cint, (Ptr{Cvoid}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        plans(kkt).jt_plan, pointer(MadNLP.nzval(kkt.jt_csc)), pointer(kkt.jt_coo.V), stream_ptr()), FactorizationException)
end

# solve_kkt! (src/IPM/factorization.jl:143-167): pre -> b2_solve -> post
function MadNLP.solve_kkt!(kkt::B200CondensedKKT{T}, w::MadNLP.AbstractKKTVector) where T
    p = plans(kkt); n = size(kkt.hess_com, 1); m = size(kkt.jt_csc, 2); wv = MadNLP.full(w)
    check(ccall((:b2_condensed_solve_pre, libb200kkt), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        p.bounds, p.jt_spmv, n, m, pointer(MadNLP.nzval(kkt.jt_csc)), pointer(kkt.pr_diag), pointer(kkt.diag_buffer),
        pointer(kkt.l_diag), pointer(kkt.u_diag), pointer(kkt.buffer), pointer(wv), stream_ptr()), SolveException)
    solve_linear_system!(kkt.linear_solver, view(wv, 1:n))
    check(ccall((:b2_condensed_solve_post, libb200kkt), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        p.bounds, p.jt_spmv, n, m, pointer(MadNLP.nzval(kkt.jt_csc)), pointer(kkt.pr_diag), pointer(kkt.diag_buffer),
        pointer(kkt.l_lower), pointer(kkt.u_lower), pointer(kkt.l_diag), pointer(kkt.u_diag), pointer(kkt.buffer), pointer(wv), stream_ptr()), SolveException)
    return w
end
solve_linear_system!(M::B200Solver{T}, x::SubArray{T,1,<:CuVector{T}}) where T =
    (check(ccall((:b2_solve, libb200kkt), Cint, (Ptr{Cvoid}, CuPtr{T}, Int32, Ptr{Cvoid}), M.handle, pointer(x), 1, stream_ptr()), SolveException); x)

# mul!(w, kkt, x, alpha, beta) (src/IPM/factorization.jl:303-324) incl. _kktmul!: ONE kernel instead of 3 SpMV + broadcasts
function MadNLP.mul!(w::MadNLP.AbstractKKTVector{T}, kkt::B200CondensedKKT{T}, x::MadNLP.AbstractKKTVector, alpha = one(T), beta = zero(T)) where T
    p = plans(kkt); n = size(kkt.hess_com, 1); m = size(kkt.jt_csc, 2)
    check(ccall((:b2_condensed_kkt_mul, libb200kkt), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T},
         Cdouble, Cdouble, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        p.bounds, p.hess_spmv, p.jt_spmv, n, m, pointer(MadNLP.nzval(kkt.hess_com)), pointer(MadNLP.nzval(kkt.jt_csc)),
        pointer(kkt.reg), pointer(kkt.du_diag), pointer(kkt.l_lower), pointer(kkt.u_lower), pointer(kkt.l_diag), pointer(kkt.u_diag),
        alpha, beta, pointer(MadNLP.full(x)), pointer(MadNLP.full(w)), stream_ptr()), SolveException)
    return w
end

# ---------------------------------------------------------------------------------------------------------------------
# Dense back-end: role of LapackCUDASolver (lib/MadNLPGPU/ext/MadNLPGPUCUDAExt/cusolver.jl:150-187), plus inertia
# ---------------------------------------------------------------------------------------------------------------------
mutable struct B200DenseSolver{T} <: AbstractLinearSolver{T}
    handle::Ptr{Cvoid}
    A::CuMatrix{T}                      # kept by reference (src/LinearSolvers/lapack.jl:40); lower triangle is read
    kkt_plan::Ptr{Cvoid}                # b2d_kkt (index sets of the DenseCondensed wrappers), created on first use
    bounds::Ptr{Cvoid}
    opt::B200Options
    logger::MadNLPLogger
end
function B200DenseSolver(A::CuMatrix{Float64}; opt = B200Options(), logger = MadNLPLogger())
    N = size(A, 1); h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:b2d_create, libb200kkt), Cint, (Int32, Int32, CuPtr{Float64}, Ptr{CB2Options}, Ptr{Ptr{Cvoid}}),
        N, stride(A, 2), pointer(A), Ref(CB2Options(opt; dense = true)), h), SymbolicException)
    M = B200DenseSolver{Float64}(h[], A, C_NULL, C_NULL, opt, logger)
    finalizer(m -> ccall((:b2d_destroy, libb200kkt), Cint, (Ptr{Cvoid},), m.handle), M)
    return M
end
factorize!(M::B200DenseSolver) = (check(ccall((:b2d_factorize, libb200kkt), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), M.handle, stream_ptr()), FactorizationException); M)
solve_linear_system!(M::B200DenseSolver{T}, x::CuVector{T}) where T =
    (check(ccall((:b2d_solve, libb200kkt), Cint, (Ptr{Cvoid}, CuPtr{T}, Int32, Ptr{Cvoid}), M.handle, pointer(x), 1, stream_ptr()), SolveException); x)
is_inertia(::B200DenseSolver) = true
function inertia(M::B200DenseSolver)
    p = Ref{Int64}(0); z = Ref{Int64}(0); n = Ref{Int64}(0)
    check(ccall((:b2d_inertia, libb200kkt), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Cvoid}), M.handle, p, z, n, stream_ptr()), FactorizationException)
    return (Int(p[]), Int(z[]), Int(n[]))
end
improve!(::B200DenseSolver) = false
introduce(M::B200DenseSolver) =
    M.opt.lapack_algorithm == MadNLP.BUNCHKAUFMAN ? "b200kkt dense LDL' (DMMA, Bunch-Kaufman pivoting)" : "b200kkt dense LDL' (DMMA, static pivoting)"
input_type(::Type{<:B200DenseSolver}) = :dense
default_options(::Type{<:B200DenseSolver}) = B200Options()
is_supported(::Type{<:B200DenseSolver}, ::Type{Float64}) = true
is_async(::B200DenseSolver) = true

const B200DenseKKT{T} = MadNLP.DenseCondensedKKTSystem{T,VT,MT,QN,LS} where {VT<:CuVector{T},MT,QN,LS<:B200DenseSolver}

function dense_plans(kkt::B200DenseKKT{T}) where T
    M = kkt.linear_solver
    if M.kkt_plan == C_NULL
        n = size(kkt.hess, 1); m = size(kkt.jac, 1); ii = Array(kkt.ind_ineq) .- 1; h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:b2d_kkt_create, libb200kkt), Cint, (Int32, Int32, Int32, Ptr{Int64}, Ptr{Ptr{Cvoid}}), n, m, length(ii), ii, h), SymbolicException)
        M.kkt_plan = h[]
        lb = Array(kkt.ind_lb) .- 1; ub = Array(kkt.ind_ub) .- 1; b = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:b2_bounds_create, libb200kkt), Cint, (Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Ptr{Cvoid}}),
            length(kkt.pr_diag), length(lb), length(ub), lb, ub, b), SymbolicException)
        M.bounds = b[]
    end
    return M.kkt_plan, M.bounds
end

# build_kkt!(::DenseCondensedKKTSystem) (src/KKT/Dense/condensed.jl:157-186): one fused DMMA SYRK + epilogue
function MadNLP.build_kkt!(kkt::B200DenseKKT{T}) where T
    n = size(kkt.hess, 1); m = size(kkt.jac, 1)
    check(ccall((:b2d_condensed_assemble, libb200kkt), Cint,
        (Int32, Int32, Int32, Int32, CuPtr{Int64}, CuPtr{Int64}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        n, m, kkt.n_ineq, kkt.n_eq, pointer(kkt.etc[:b200_ind_ineq0]), pointer(kkt.etc[:b200_ind_eq0]), pointer(kkt.hess), pointer(kkt.jac),
        pointer(kkt.pr_diag), pointer(kkt.du_diag), pointer(kkt.diag_buffer), pointer(kkt.aug_com), stream_ptr()), FactorizationException)
end
# (kkt.etc is the Dict{Symbol,Any} scratch slot of the struct, Dense/condensed.jl:49: the 0-based device copies of ind_ineq / ind_eq
#  are stored there once:  kkt.etc[:b200_ind_ineq0] = CuVector(kkt.ind_ineq .- 1) ...)

# solve_kkt!(::DenseCondensedKKTSystem) (src/IPM/factorization.jl:190-229)
function MadNLP.solve_kkt!(kkt::B200DenseKKT{T}, w::MadNLP.AbstractKKTVector) where T
    kp, bp = dense_plans(kkt); wv = MadNLP.full(w)
    check(ccall((:b2d_kkt_solve_pre, libb200kkt), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        kp, bp, pointer(kkt.jac), pointer(kkt.pr_diag), pointer(kkt.diag_buffer), pointer(kkt.l_diag), pointer(kkt.u_diag),
        pointer(kkt.buffer), pointer(kkt.pd_buffer), pointer(wv), stream_ptr()), SolveException)
    solve_linear_system!(kkt.linear_solver, kkt.pd_buffer)
    check(ccall((:b2d_kkt_solve_post, libb200kkt), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        kp, bp, pointer(kkt.jac), pointer(kkt.pr_diag), pointer(kkt.diag_buffer), pointer(kkt.l_lower), pointer(kkt.u_lower),
        pointer(kkt.l_diag), pointer(kkt.u_diag), pointer(kkt.buffer), pointer(kkt.pd_buffer), pointer(wv), stream_ptr()), SolveException)
    return w
end

# mul!(w, ::AbstractDenseKKTSystem, x, alpha, beta) (src/IPM/factorization.jl:303-324)
function MadNLP.mul!(w::MadNLP.AbstractKKTVector{T}, kkt::B200DenseKKT{T}, x::MadNLP.AbstractKKTVector, alpha = one(T), beta = zero(T)) where T
    kp, bp = dense_plans(kkt)
    check(ccall((:b2d_kkt_mul, libb200kkt), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Cdouble, Cdouble, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        kp, bp, pointer(kkt.hess), pointer(kkt.jac), pointer(kkt.reg), pointer(kkt.du_diag), pointer(kkt.l_lower), pointer(kkt.u_lower),
        pointer(kkt.l_diag), pointer(kkt.u_diag), alpha, beta, pointer(MadNLP.full(x)), pointer(MadNLP.full(w)), stream_ptr()), SolveException)
    return w
end

# ---------------------------------------------------------------------------------------------------------------------
# Optional: the vector passes of RichardsonIterator (src/LinearSolvers/backsolve.jl:36-52) as single launches.
#   b200_richardson_begin!(b, w, x, norms)   norms[3] = ||b||_inf ; x = 0 ; w = b
#   b200_richardson_update!(b, w, x, norms)  x += w ; w = b ; norms[1] = 0 ; norms[2] = ||x||_inf
# followed by mul!(w, kkt, x, -1, 1) through b2_condensed_kkt_mul_norm (accumulates ||w||_inf into norms[1]); one
# 24-byte D2H copy then carries the three norms of the stopping rule.
# ---------------------------------------------------------------------------------------------------------------------
function b200_richardson_begin!(b::CuVector{T}, w::CuVector{T}, x::CuVector{T}, norms::CuVector{T}) where T
    check(ccall((:b2_richardson_begin, libb200kkt), Cint, (Int64, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        length(b), pointer(b), pointer(w), pointer(x), pointer(norms, 3), stream_ptr()), SolveException)
end
function b200_richardson_update!(b::CuVector{T}, w::CuVector{T}, x::CuVector{T}, norms::CuVector{T}) where T
    check(ccall((:b2_richardson_update, libb200kkt), Cint, (Int64, CuPtr{T}, CuPtr{T}, CuPtr{T}, CuPtr{T}, Ptr{Cvoid}),
        length(b), pointer(b), pointer(w), pointer(x), pointer(norms), stream_ptr()), SolveException)
end

# inertia read split in two (queue more work behind factorize!, block once): b2_inertia_enqueue / b2_inertia_fetch
inertia_enqueue!(M::B200Solver) = check(ccall((:b2_inertia_enqueue, libb200kkt), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), M.handle, stream_ptr()), FactorizationException)
function inertia_fetch(M::B200Solver)
    p = Ref{Int64}(0); z = Ref{Int64}(0); n = Ref{Int64}(0)
    check(ccall((:b2_inertia_fetch, libb200kkt), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}), M.handle, p, z, n), FactorizationException)
    return (Int(p[]), Int(z[]), Int(n[]))
end

end # module
