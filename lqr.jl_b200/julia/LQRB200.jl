# LQRB200.jl — `ccall`-only Julia shim over liblqrb200.so (include/lqrb200.h).
#
# STATUS: static artefact.  Julia is not installed in the build image or on the GPU box, so this file has never
# been executed; the executable tests drive the same C ABI from Python (ctypes) and from plain C
# (tests/abi_smoke.c), and tests/test_host_cpu.py::test_julia_shim_binds_every_header_symbol checks that every
# entry point of the header is bound here with the argument count the header declares.
#
# It re-exposes LQR.jl's hot path UNDER THE REFERENCE'S OWN NAMES, so that `using LQRB200` in place of `using LQR`
# swaps the path (SURVEY §8b).  Every type carries a trailing batch axis; a single-instance call is batch = 1.
#
#   reference (bjack205/LQR.jl)                                        this shim
#   LQRProblem, size, num_vars        src/lqr_problem.jl:1-25           LQRProblem, Base.size, num_vars
#   DPSolver, solve!                  src/dynamic_programming.jl:8-72   DPSolver, solve!(sol, solver, prob)
#   rollout!                          src/least_squares.jl:195-202      rollout!
#   BlockCholesky, cholesky!, ldiv!,\ src/block_cholesky.jl:19-101      BlockCholesky, cholesky!, ldiv!, \
#   InvertedQuadratic, update_cost!,  src/block_cholesky.jl:107-159     InvertedQuadratic, update_cost!,
#     update_cholesky!, gradient                                          update_cholesky!, gradient
#   ConstraintBlock(s), dims,         src/conblocks.jl:36-113           ConstraintBlock, ConstraintBlocks, dims,
#     copy_blocks!                                                        copy_blocks!
#   build_shur_factors,               src/jacobian_blocks.jl:155-229    build_shur_factors,
#     calculate_shur_factors!,                                            calculate_shur_factors!,
#     copy_shur_factors!              src/jacobian_blocks.jl:173-211      copy_shur_factors!
#   cholesky!(U, F),                  src/cholesky_solve.jl:28-143      cholesky!(U, F), forward_substitution!,
#     forward_/backward_substitution!                                     backward_substitution!
#   CholeskySolver, _solve!, solve!,  src/cholesky_solver.jl:39-273     CholeskySolver, _solve!, solve!, step!,
#     step!, update!, calculate_primals!, residual,                       update!, calculate_primals!, residual,
#     second_order_correction!, get_*                                     second_order_correction!, get_*
#
# Arrays are ordinary Julia `Array{Float64}` whose LAST axis is the batch: A is n×n×(N-1)×batch.  That is exactly
# the ABI's "instance-major" layout, so no copies are made on the Julia side; the library moves the data to the
# GPU, repacks it batch-minor, solves, and writes the results back.  Device-resident use (no host copies) goes
# through the `*_packed!` wrappers at the end, which take raw device pointers.
module LQRB200

using LinearAlgebra

const lib = get(ENV, "LQRB200_LIB", joinpath(@__DIR__, "..", "liblqrb200.so"))

const HESS_DENSE, HESS_BLOCKDIAG, HESS_DIAG = Int32(0), Int32(1), Int32(2)
const FLAG_SOC, FLAG_LTI, FLAG_NO_AFFINE, FLAG_WARM_START = Int32(1), Int32(2), Int32(4), Int32(8)
const DevPtr = Ptr{Float64}   # a device address (e.g. `pointer(::CuArray{Float64})` reinterpreted by the caller)

struct LQRBError <: Exception
    code::Int32
    msg::String
end

# ------------------------------------------------------------------ handle -------------------------------
mutable struct Handle
    ptr::Ptr{Cvoid}
    function Handle(device::Integer=0)
        ref = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:lqrb_create, lib), Int32, (Ref{Ptr{Cvoid}}, Int32), ref, device)
        rc == 0 || throw(LQRBError(rc, "lqrb_create failed (an sm_100 GPU is required; there is no CPU fallback)"))
        h = new(ref[])
        finalizer(h -> ccall((:lqrb_destroy, lib), Int32, (Ptr{Cvoid},), h.ptr), h)
        return h
    end
end

function check(h::Handle, rc::Integer)
    rc == 0 && return nothing
    msg = unsafe_string(ccall((:lqrb_last_error_string, lib), Cstring, (Ptr{Cvoid},), h.ptr))
    throw(LQRBError(Int32(rc), msg))
end

version() = ccall((:lqrb_version, lib), Int32, ())
function device_count()
    c = Ref{Int32}(0)
    ccall((:lqrb_device_count, lib), Int32, (Ref{Int32},), c)
    return Int(c[])
end
"order all work of the handle on a caller-owned cudaStream_t (C_NULL: the handle's own stream)"
set_stream!(h::Handle, stream::Ptr{Cvoid}) = check(h, ccall((:lqrb_set_stream, lib), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), h.ptr, stream))
synchronize(h::Handle) = check(h, ccall((:lqrb_synchronize, lib), Int32, (Ptr{Cvoid},), h.ptr))
launch_count(h::Handle) = ccall((:lqrb_launch_count, lib), Int64, (Ptr{Cvoid},), h.ptr)
last_kernel_name(h::Handle) = unsafe_string(ccall((:lqrb_last_kernel_name, lib), Cstring, (Ptr{Cvoid},), h.ptr))
set_option!(h::Handle, name::AbstractString, value::Integer) =
    check(h, ccall((:lqrb_set_option, lib), Int32, (Ptr{Cvoid}, Cstring, Int64), h.ptr, name, value))
"measured FP64 peak of the device in TFLOP/s (kind 0: DFMA, 1: DMMA)"
function fp64_peak(h::Handle, kind::Integer=1; seconds::Real=0.4)
    t = Ref{Float64}(0.0)
    check(h, ccall((:lqrb_fp64_peak_f64, lib), Int32, (Ptr{Cvoid}, Int32, Float64, Ref{Float64}), h.ptr, kind, seconds, t))
    return t[]
end

"(log2 pivot ratios of the last tuned KKT launch, instances re-solved by the Cholesky-based kernel)"
function kkt_last_condition(h::Handle, count::Integer)
    out = zeros(Int32, count)
    n = Ref{Int64}(0)
    check(h, ccall((:lqrb_kkt_last_condition, lib), Int32, (Ptr{Cvoid}, Int64, Ptr{Int32}, Ref{Int64}), h.ptr, count, out, n))
    return out, n[]
end

ptr_or_null(a::Nothing) = Ptr{Float64}(C_NULL)
ptr_or_null(a::Array{Float64}) = pointer(a)
iptr_or_null(a::Nothing) = Ptr{Int32}(C_NULL)
iptr_or_null(a::Array{Int32}) = pointer(a)

# ------------------------------------------------------------------ layout queries -----------------------
padded_batch(batch::Integer) = ccall((:lqrb_padded_batch, lib), Int64, (Int64,), batch)
num_vars(n::Integer, m::Integer, N::Integer) = ccall((:lqrb_num_vars, lib), Int64, (Int32, Int32, Int32), n, m, N)
num_cons(n::Integer, N::Integer, p::Vector{Int32}) = ccall((:lqrb_num_cons, lib), Int64, (Int32, Int32, Ptr{Int32}), n, N, p)
struct RiccatiLayout
    rows_per_knot::Int64
    knot_count::Int64
    term_rows::Int64
    z_rows::Int64
    gain_rows::Int64
end
function riccati_layout(n, m, N, flags=Int32(0))
    out = Ref(RiccatiLayout(0, 0, 0, 0, 0))
    rc = ccall((:lqrb_riccati_layout, lib), Int32, (Int32, Int32, Int32, Int32, Ref{RiccatiLayout}), n, m, N, flags, out)
    rc == 0 || throw(LQRBError(rc, "lqrb_riccati_layout: bad argument $(-rc)"))
    return out[]
end
kkt_data_rows(n, m, N, p::Vector{Int32}, hess_mode, explicit_d2=false) =
    ccall((:lqrb_kkt_data_rows, lib), Int64, (Int32, Int32, Int32, Ptr{Int32}, Int32, Int32), n, m, N, p, hess_mode, explicit_d2)
kkt_knot_offset(n, m, N, p::Vector{Int32}, hess_mode, explicit_d2, k) =
    ccall((:lqrb_kkt_knot_offset, lib), Int64, (Int32, Int32, Int32, Ptr{Int32}, Int32, Int32, Int32), n, m, N, p, hess_mode, explicit_d2, k)
riccati_tile_width(h::Handle, n, m) = ccall((:lqrb_riccati_tile_width, lib), Int32, (Ptr{Cvoid}, Int32, Int32), h.ptr, n, m)
kkt_tile_width(h::Handle, n, m, N, p::Vector{Int32}, hess_mode, explicit_d2=false) =
    ccall((:lqrb_kkt_tile_width, lib), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ptr{Int32}, Int32, Int32), h.ptr, n, m, N, p, hess_mode, explicit_d2)

# ------------------------------------------------------------------ LQRProblem (src/lqr_problem.jl:1-25) --
"Batched LQRProblem: the reference's fields (Qf, Q, R, A, B, x0, u0, tf, N) with a trailing batch axis.  A 3-D `A`
(n×n×batch) is the reference's time-invariant form; a 4-D `A` (n×n×(N-1)×batch) is the per-knot generalisation;
`q`, `r`, `qf` add affine cost terms (SURVEY Appendix A)."
struct LQRProblem
    Qf::Array{Float64,3}   # n×n×batch
    Q::Array{Float64}      # n×n×batch (LTI) or n×n×(N-1)×batch (LTV)
    R::Array{Float64}
    A::Array{Float64}
    B::Array{Float64}
    x0::Matrix{Float64}    # n×batch
    u0::Matrix{Float64}    # m×batch
    tf::Float64
    N::Int
    q::Union{Nothing,Array{Float64}}
    r::Union{Nothing,Array{Float64}}
    qf::Union{Nothing,Matrix{Float64}}
end
LQRProblem(Qf, Q, R, A, B, x0, u0, tf, N) = LQRProblem(Qf, Q, R, A, B, x0, u0, tf, N, nothing, nothing, nothing)
islti(p::LQRProblem) = ndims(p.A) == 3
Base.size(p::LQRProblem) = (size(p.A, 1), size(p.B, 2), p.N)
batchsize(p::LQRProblem) = size(p.x0, 2)
num_vars(p::LQRProblem) = ((n, m, N) = size(p); Int(num_vars(n, m, N)))

"Primals-ordered solution Z = [x1;u1;…;xN] per instance (src/lqr_problem.jl:46-73) + gains"
struct LQRSolution
    Z::Matrix{Float64}           # NN×batch
    K::Array{Float64,4}          # m×n×(N-1)×batch
    d::Array{Float64,3}          # m×(N-1)×batch (feed-forward; zero for the reference's DPSolver form)
    info::Vector{Int32}
end
function LQRSolution(prob::LQRProblem)
    n, m, N = size(prob); b = batchsize(prob)
    LQRSolution(zeros(num_vars(prob), b), zeros(m, n, N - 1, b), zeros(m, N - 1, b), zeros(Int32, b))
end
"state k of instance i as a view (the reference's sol.X[k])"
state(sol::LQRSolution, n, m, k, i=1) = view(sol.Z, (k - 1) * (n + m) .+ (1:n), i)
control(sol::LQRSolution, n, m, k, i=1) = view(sol.Z, (k - 1) * (n + m) + n .+ (1:m), i)

# ------------------------------------------------------------------ DPSolver (src/dynamic_programming.jl) -
struct DPSolver
    handle::Handle
end
DPSolver(prob::LQRProblem; device=0) = DPSolver(Handle(device))

"solve!(sol, solver::DPSolver, prob): src/dynamic_programming.jl:54-72 (compute_gain! :37-43, compute_ctg! :48-52)"
function solve!(sol::LQRSolution, solver::DPSolver, prob::LQRProblem)
    n, m, N = size(prob)
    flags = islti(prob) ? FLAG_LTI : Int32(0)
    GC.@preserve sol prob begin
        rc = ccall((:lqrb_riccati_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Int32,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            solver.handle.ptr, n, m, N, batchsize(prob), flags,
            prob.A, prob.B, prob.Q, prob.R, ptr_or_null(prob.q), ptr_or_null(prob.r),
            prob.Qf, ptr_or_null(prob.qf), prob.x0, sol.Z, sol.K, sol.d, sol.info)
    end
    check(solver.handle, rc)
    return sol
end

"rollout!(X, U, prob): X[:,1,i] = x0; X[:,k+1,i] = A X[:,k,i] + B U[:,k,i]  (src/least_squares.jl:195-202)"
function rollout!(X::Array{Float64,3}, U::Array{Float64,3}, prob::LQRProblem, handle::Handle)
    n, m, N = size(prob)
    flags = islti(prob) ? FLAG_LTI : Int32(0)
    GC.@preserve X U prob begin
        rc = ccall((:lqrb_rollout_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
            handle.ptr, n, m, N, batchsize(prob), flags, prob.A, prob.B, prob.x0, U, X)
    end
    check(handle, rc)
    return X
end

"""riccati_grad!(G, prob, Z, dZ, handle): gradients of a loss l(Z) through solve!(sol, ::DPSolver, prob) from
dZ = dl/dZ (NN×batch).  G is a NamedTuple (A, B, Q, R, q, r, Qf, qf, x0) of arrays shaped like the problem's (any may
be `nothing`); returns the potrf info of the adjoint solve per instance."""
function riccati_grad!(G::NamedTuple, prob::LQRProblem, Z::Matrix{Float64}, dZ::Matrix{Float64}, handle::Handle)
    n, m, N = size(prob)
    flags = islti(prob) ? FLAG_LTI : Int32(0)
    info = zeros(Int32, batchsize(prob))
    g(x) = x === nothing ? C_NULL : pointer(x)
    GC.@preserve G prob Z dZ info begin
        rc = ccall((:lqrb_riccati_grad_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Int32}),
            handle.ptr, n, m, N, batchsize(prob), flags, prob.A, prob.B, prob.Q, prob.R, ptr_or_null(prob.q),
            ptr_or_null(prob.r), prob.Qf, ptr_or_null(prob.qf), Z, dZ, g(G.A), g(G.B), g(G.Q), g(G.R), g(G.q), g(G.r),
            g(G.Qf), g(G.qf), g(G.x0), info)
    end
    check(handle, rc)
    return info
end

"""riccati_grad_gains!(G, prob, Z, dZ, dK, dkff, handle): gradients of a loss l(Z, K, kff) through
solve!(sol, ::DPSolver, prob), the gains included, from dZ = dl/dZ (NN×batch), dK = dl/dK (m×n×(N-1)×batch) and
dkff = dl/dkff (m×(N-1)×batch).  Any cotangent may be `nothing`, not all three (Z is read only with dZ).  G as in
riccati_grad!; returns the info of the solve per instance."""
function riccati_grad_gains!(G::NamedTuple, prob::LQRProblem, Z::Union{Nothing,Matrix{Float64}},
                             dZ::Union{Nothing,Matrix{Float64}}, dK::Union{Nothing,Array{Float64,4}},
                             dkff::Union{Nothing,Array{Float64,3}}, handle::Handle)
    n, m, N = size(prob)
    flags = islti(prob) ? FLAG_LTI : Int32(0)
    info = zeros(Int32, batchsize(prob))
    g(x) = x === nothing ? C_NULL : pointer(x)
    GC.@preserve G prob Z dZ dK dkff info begin
        rc = ccall((:lqrb_riccati_grad_gains_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            handle.ptr, n, m, N, batchsize(prob), flags, prob.A, prob.B, prob.Q, prob.R, ptr_or_null(prob.q),
            ptr_or_null(prob.r), prob.Qf, ptr_or_null(prob.qf), g(Z), g(dZ), g(dK), g(dkff), g(G.A), g(G.B), g(G.Q),
            g(G.R), g(G.q), g(G.r), g(G.Qf), g(G.qf), g(G.x0), info)
    end
    check(handle, rc)
    return info
end

"""dare!(P, K, A, B, Q, R, handle): stabilising solution P (n×n×batch) and stationary gain K (m×n×batch, u = -K x) of
the discrete algebraic Riccati equation of A (n×n×batch), B (n×m×batch), Q (n×n×batch), R (m×m×batch) by structured
doubling.  P or K may be `nothing`, not both.  Returns (info, iters) per instance (include/lqrb200.h codes)."""
function dare!(P::Union{Nothing,Array{Float64,3}}, K::Union{Nothing,Array{Float64,3}}, A::Array{Float64,3},
               B::Array{Float64,3}, Q::Array{Float64,3}, R::Array{Float64,3}, handle::Handle)
    n, m, batch = size(A, 1), size(B, 2), size(A, 3)
    info = zeros(Int32, batch)
    iters = zeros(Int32, batch)
    g(x) = x === nothing ? C_NULL : pointer(x)
    GC.@preserve P K A B Q R info iters begin
        rc = ccall((:lqrb_dare_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
            handle.ptr, n, m, batch, A, B, Q, R, g(P), g(K), iters, info)
    end
    check(handle, rc)
    return info, iters
end

"""dare_grad!(G, A, B, R, P, dP, dK, handle): gradients of a loss l(P, K) through dare! from dP = dl/dP (n×n×batch)
and dK = dl/dK (m×n×batch), either may be `nothing`, not both.  G is a NamedTuple (A, B, Q, R) of arrays shaped like
the inputs (any may be `nothing`); returns the info per instance."""
function dare_grad!(G::NamedTuple, A::Array{Float64,3}, B::Array{Float64,3}, R::Array{Float64,3}, P::Array{Float64,3},
                    dP::Union{Nothing,Array{Float64,3}}, dK::Union{Nothing,Array{Float64,3}}, handle::Handle)
    n, m, batch = size(A, 1), size(B, 2), size(A, 3)
    info = zeros(Int32, batch)
    g(x) = x === nothing ? C_NULL : pointer(x)
    GC.@preserve G A B R P dP dK info begin
        rc = ccall((:lqrb_dare_grad_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            handle.ptr, n, m, batch, A, B, R, P, g(dP), g(dK), g(G.A), g(G.B), g(G.Q), g(G.R), info)
    end
    check(handle, rc)
    return info
end

"""admm_cache!(cache, A, B, Q, R, rho, handle): the cache of box-constrained MPC by ADMM (lqrb_admm_cache_f64) for
A (n×n×batch), B (n×m×batch), Q (n×n×batch), R (m×m×batch) and rho > 0: cache is (4n²+2nm+2m²+1)×batch, per instance
[A | B | Q | R | Qf | K | C1 | C2 | rho] with the terminal cost Qf = P̃ - rho I of the solve.  Returns the info per
instance (the DARE's codes)."""
function admm_cache!(cache::Matrix{Float64}, A::Array{Float64,3}, B::Array{Float64,3}, Q::Array{Float64,3},
                     R::Array{Float64,3}, rho::Float64, handle::Handle)
    n, m, batch = size(A, 1), size(B, 2), size(A, 3)
    info = zeros(Int32, batch)
    GC.@preserve cache A B Q R info begin
        rc = ccall((:lqrb_admm_cache_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int64, Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Int32}),
            handle.ptr, n, m, batch, rho, A, B, Q, R, cache, info)
    end
    check(handle, rc)
    return info
end

"lqrb_admm_options_t"
struct AdmmOptions
    max_iter::Int32
    eps_pri::Float64
    eps_dual::Float64
end

"""admm_solve!(Z, cache, x0, bounds, handle; N, xref, uref, state, warm, max_iter, eps): box-constrained MPC by ADMM
(lqrb_admm_solve_f64) on a cache from admm_cache!.  Z is (N n + (N-1) m)×batch in Primals order; bounds is a NamedTuple
(umin, umax, xmin, xmax) of m×(N-1)×batch / n×(N-1)×batch arrays or `nothing` (±Inf); xref (n×N×batch), uref
(m×(N-1)×batch) may be `nothing` (0); state (2(N-1)(m+n)×batch) is read when warm and written when given.  Returns
(info, iters, res) per instance."""
function admm_solve!(Z::Matrix{Float64}, cache::Matrix{Float64}, x0::Matrix{Float64}, bounds::NamedTuple,
                     handle::Handle; N::Integer, m::Integer, xref=nothing, uref=nothing,
                     state::Union{Nothing,Matrix{Float64}}=nothing, warm::Bool=false, max_iter::Integer=100,
                     eps::Float64=1e-6)
    n, batch = size(x0, 1), size(x0, 2)
    info = zeros(Int32, batch)
    iters = zeros(Int32, batch)
    res = zeros(Float64, 2, batch)
    opts = Ref(AdmmOptions(Int32(max_iter), eps, eps))
    g(x) = x === nothing ? C_NULL : pointer(x)
    GC.@preserve Z cache x0 bounds xref uref state info iters res opts begin
        rc = ccall((:lqrb_admm_solve_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Int32, Ref{AdmmOptions}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Int32}, Ptr{Float64}, Ptr{Int32}),
            handle.ptr, n, m, N, batch, warm ? FLAG_WARM_START : Int32(0), opts, cache, x0, g(xref), g(uref),
            g(bounds.umin), g(bounds.umax), g(bounds.xmin), g(bounds.xmax), g(state), Z, iters, res, info)
    end
    check(handle, rc)
    return info, iters, res
end

# ------------------------------------------------------------------ LeastSquaresSolver (src/least_squares.jl)
"LeastSquaresSolver(prob): the condensed (block-Toeplitz) form of the unconstrained LTI problem, src/least_squares.jl:1-59"
struct LeastSquaresSolver
    handle::Handle
    info::Vector{Int32}
end
LeastSquaresSolver(prob::LQRProblem; device=0) = LeastSquaresSolver(Handle(device), zeros(Int32, batchsize(prob)))
"solve!(sol, solver::LeastSquaresSolver, prob): src/least_squares.jl:158-190 ((T'QT + R) U = -T'Q L x0 by Cholesky, rollout!)"
function solve!(sol::LQRSolution, solver::LeastSquaresSolver, prob::LQRProblem)
    islti(prob) || throw(ArgumentError("LeastSquaresSolver takes the time-invariant LQRProblem"))
    n, m, N = size(prob)
    GC.@preserve sol prob solver begin
        rc = ccall((:lqrb_lsq_solve_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            solver.handle.ptr, n, m, N, batchsize(prob), prob.A, prob.B, prob.Q, prob.R, prob.Qf, prob.x0, sol.Z, solver.info)
    end
    check(solver.handle, rc)
    return sol
end

# ------------------------------------------------------------------ BlockCholesky (src/block_cholesky.jl) -
struct BlockCholesky
    handle::Handle
    M::Array{Float64,3}     # (n+m)×(n+m)×batch: upper factor, or reciprocals on the diagonal (diag mode)
    n::Int
    m::Int
    mode::Int32
    uplo::Char
    info::Vector{Int32}
end
"BlockCholesky(n, m; diag, block_diag, uplo): src/block_cholesky.jl:19-52 (only uplo = 'U', the reference's default)"
function BlockCholesky(handle::Handle, n::Int, m::Int, batch::Int=1; diag=false, block_diag=false, uplo::Char='U')
    uplo == 'U' || throw(ArgumentError("only uplo = 'U' is supported"))
    mode = diag ? HESS_DIAG : (block_diag ? HESS_BLOCKDIAG : HESS_DENSE)
    BlockCholesky(handle, zeros(n + m, n + m, batch), n, m, mode, uplo, zeros(Int32, batch))
end

"cholesky!(chol, A, B[, C]): src/block_cholesky.jl:55-91"
function LinearAlgebra.cholesky!(chol::BlockCholesky, A::Array{Float64,3}, B::Array{Float64,3},
                                 C::Union{Nothing,Array{Float64,3}}=nothing)
    GC.@preserve chol A B C begin
        rc = ccall((:lqrb_block_cholesky_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            chol.handle.ptr, chol.n, chol.m, size(chol.M, 3), chol.mode, A, B, ptr_or_null(C), chol.M, chol.info)
    end
    check(chol.handle, rc)
    return chol
end

"ldiv!(chol, b): src/block_cholesky.jl:93-96; b is (n+m)×nrhs×batch"
function LinearAlgebra.ldiv!(chol::BlockCholesky, b::Array{Float64,3})
    GC.@preserve chol b begin
        rc = ccall((:lqrb_block_ldiv_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int64, Int32, Ptr{Float64}, Int32, Ptr{Float64}),
            chol.handle.ptr, chol.n, chol.m, size(chol.M, 3), chol.mode, chol.M, size(b, 2), b)
    end
    check(chol.handle, rc)
    return b
end
Base.:\(chol::BlockCholesky, b::Array{Float64,3}) = ldiv!(chol, copy(b))

# ------------------------------------------------------------------ InvertedQuadratic (src/block_cholesky.jl:107-159)
"chol(H_k) + gradient (q, r) of one knot's cost expansion, batched"
struct InvertedQuadratic
    chol::BlockCholesky
    q::Matrix{Float64}   # n×batch
    r::Matrix{Float64}   # m×batch
end
InvertedQuadratic(handle::Handle, n::Int, m::Int, batch::Int=1; diag=false, block_diag=true) =
    InvertedQuadratic(BlockCholesky(handle, n, m, batch; diag=diag, block_diag=block_diag), zeros(n, batch), zeros(m, batch))

"update_cost!(icost, Q, R, q, r[, H]): src/block_cholesky.jl:145-153 (the cost is passed as its blocks)"
function update_cost!(icost::InvertedQuadratic, Q::Array{Float64,3}, R::Array{Float64,3}, q, r, H=nothing)
    if icost.chol.mode != HESS_DENSE || H === nothing
        cholesky!(icost.chol, Q, R)
    else
        cholesky!(icost.chol, Q, R, H)
    end
    icost.q .= q
    icost.chol.m > 0 && (icost.r .= r)
    return icost
end
"update_cholesky!(chols, costs): src/block_cholesky.jl:155-159; costs[k] = (Q=, R=, q=, r=[, H=])"
function update_cholesky!(chols::Vector{InvertedQuadratic}, costs)
    for k in eachindex(chols)
        c = costs[k]
        update_cost!(chols[k], c.Q, c.R, c.q, c.r, get(c, :H, nothing))
    end
end
"gradient(icost): [q; r], or q at the terminal knot (src/block_cholesky.jl:126-132)"
gradient(icost::InvertedQuadratic) = icost.chol.m > 0 ? vcat(icost.q, icost.r) : copy(icost.q)

# ------------------------------------------------------------------ ConstraintBlock (src/conblocks.jl:36-113)
"Y = [D2; C; D1] ((n1+p+n2)×w×batch), y = [c; d], with views that alias Y and y like the reference's"
struct ConstraintBlock
    y::Matrix{Float64}
    Y::Array{Float64,3}
    res::Matrix{Float64}
    D2::SubArray
    C::SubArray
    D1::SubArray
    c::SubArray
    d::SubArray
end
function ConstraintBlock(n1::Int, p::Int, n2::Int, w::Int, batch::Int=1)
    y = zeros(p + n2, batch)
    Y = zeros(n1 + p + n2, w, batch)
    ConstraintBlock(y, Y, zeros(w, batch), view(Y, 1:n1, :, :), view(Y, n1 .+ (1:p), :, :), view(Y, (n1 + p) .+ (1:n2), :, :),
                    view(y, 1:p, :), view(y, p .+ (1:n2), :))
end
"dims(block) = (n1, p, n2): src/conblocks.jl:98"
dims(block::ConstraintBlock) = size(block.D2, 1), size(block.C, 1), size(block.D1, 1)
"per-knot block sizes of a dynamics-coupled problem (src/conblocks.jl:74-96); D2 starts as the structural [-I 0]"
function ConstraintBlocks(n::Int, m::Int, N::Int, p::Vector{Int32}, batch::Int=1)
    map(1:N) do k
        blk = ConstraintBlock(k > 1 ? n : 0, Int(p[k]), k < N ? n : 0, n + m * (k < N), batch)
        for i = 1:(k > 1 ? n : 0)
            blk.D2[i, i, :] .= -1.0
        end
        blk
    end
end
"copy_blocks!(D, d, blocks[, i]): src/conblocks.jl:100-113 for instance i"
function copy_blocks!(D, d, blocks::Vector{ConstraintBlock}, i::Int=1)
    off1 = off2 = 0
    for block in blocks
        n1, p, n2 = dims(block)
        w = size(block.Y, 2)
        D[off1 .+ (1:n1+p+n2), off2 .+ (1:w)] .= view(block.Y, :, :, i)
        d[off1 + n1 .+ (1:p+n2)] .= view(block.y, :, i)
        off1 += n1 + p
        off2 += w
    end
    return D, d
end

"gen_con_inds(cons, N, structure): src/conblocks.jl:122-166.  `cons` stands in for TrajOptCore's ConstraintList: a vector
of (length, knots::UnitRange) pairs; returns cons[i][j] = index range of constraint i at its j-th knot."
function gen_con_inds(cons::Vector{<:Tuple{Int,UnitRange{Int}}}, N::Int, structure::Symbol=:by_knotpoint)
    out = [[1:0 for _ in knots] for (_, knots) in cons]
    if structure == :by_constraint
        idx = 0
        for (i, (len, knots)) in enumerate(cons), j in eachindex(knots)
            out[i][j] = idx .+ (1:len); idx += len
        end
    elseif structure == :by_knotpoint
        idx = 0
        for k = 1:N, (i, (len, knots)) in enumerate(cons)
            if k in knots
                out[i][k - first(knots) + 1] = idx .+ (1:len); idx += len
            end
        end
    elseif structure == :by_block
        idx = zeros(Int, N)
        for k = 1:N, (i, (len, knots)) in enumerate(cons)
            if k in knots
                out[i][k - first(knots) + 1] = idx[k] .+ (1:len); idx[k] += len
            end
        end
    else
        throw(ArgumentError("unknown structure $structure"))
    end
    return out
end

# ------------------------------------------------------------------ CholeskySolver (src/cholesky_solver.jl)
# The reference fills Jinv / conSet.blocks through TrajOptCore (update!, :155-164).  A batched caller supplies a
# `linearize!(solver)` callback that writes the same linearised blocks (Q, R, Hux, q, r, A, B, d, C, c) as plain
# arrays with a trailing batch axis; everything after that point runs on the GPU.

"Names the device-resident block rows (Vector{BlockUpperTriangular3}, src/jacobian_blocks.jl:95-169) for the step
functions: kind = :shur (S before factorisation) or :chol (block rows of U)"
struct ShurBlocks
    solver::Any
    kind::Symbol
end

mutable struct CholeskySolver
    handle::Handle
    n::Int; m::Int; N::Int
    p::Vector{Int32}             # stage-constraint rows per knot (src/conblocks.jl:74-96)
    hess_mode::Int32
    Q::Array{Float64,4}; R::Array{Float64,4}; Hux::Union{Nothing,Array{Float64,4}}
    q::Array{Float64,3}; r::Array{Float64,3}
    A::Array{Float64,4}; B::Array{Float64,4}; d::Array{Float64,3}
    D2::Union{Nothing,Matrix{Float64}}     # nothing ⇒ [-I 0]
    C::Matrix{Float64}; c::Matrix{Float64} # concatenated blocks × batch
    δZ::Matrix{Float64}; λ::Matrix{Float64}; res::Matrix{Float64}; info::Vector{Int32}
    Z::Matrix{Float64}                     # current iterate (Primals order) for solve!/step!
    linearize!::Union{Nothing,Function}    # update!: fills the blocks above from solver.Z
    max_violation::Union{Nothing,Function} # feas_p of step! (src/cholesky_solver.jl:126)
    Ginv::Bool
    factored::Bool
    shur_blocks::ShurBlocks
    chol_blocks::ShurBlocks
    function CholeskySolver(handle::Handle, n, m, N, p::Vector{Int32}, hess_mode, Q, R, Hux, q, r, A, B, d, D2, C, c;
                            linearize! = nothing, max_violation = nothing)
        b = size(q, 3)
        NN, P = Int(num_vars(n, m, N)), Int(num_cons(n, N, p))
        s = new(handle, n, m, N, p, Int32(hess_mode), Q, R, Hux, q, r, A, B, d, D2, C, c,
                zeros(NN, b), zeros(P, b), zeros(NN, b), zeros(Int32, b), zeros(NN, b), linearize!, max_violation, true, false)
        s.shur_blocks = ShurBlocks(s, :shur)
        s.chol_blocks = ShurBlocks(s, :chol)
        return s
    end
end
Base.size(s::CholeskySolver) = (s.n, s.m, s.N)
num_vars(s::CholeskySolver) = size(s.δZ, 1)
batchsize(s::CholeskySolver) = size(s.δZ, 2)
_flags(s::CholeskySolver) = s.Ginv ? Int32(0) : FLAG_SOC

"build_shur_factors(solver, :U): src/jacobian_blocks.jl:155-169 (only the upper variant has substitution methods)"
function build_shur_factors(s::CholeskySolver, uplo::Symbol=:U)
    uplo == :U || throw(ArgumentError("only :U is supported (src/cholesky_solve.jl:145-168)"))
    return ShurBlocks(s, :shur)
end

function _call_kkt!(s::CholeskySolver, flags::Int32)
    GC.@preserve s begin
        rc = ccall((:lqrb_kkt_solve_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32, Int32,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            s.handle.ptr, s.n, s.m, s.N, batchsize(s), s.p, s.hess_mode, flags,
            s.Q, s.R, ptr_or_null(s.Hux), s.q, s.r, s.A, s.B, s.d, ptr_or_null(s.D2), s.C, s.c,
            s.δZ, s.λ, s.res, s.info)
    end
    check(s.handle, rc)
    return s
end

"""kkt_grad!(G, solver, dZ̄, λ̄): gradients of a loss l(δZ, λ) through the last _solve!(solver) (δZ, λ as it left
them) from dZ̄ = dl/dδZ (NN×batch) and λ̄ = dl/dλ (P×batch); either may be `nothing`, not both.  G is a NamedTuple
(Q, R, Hux, q, r, A, B, d, D2, C, c) of arrays shaped like the solver's (any may be `nothing`); returns the potrf info
of the adjoint solve per instance."""
function kkt_grad!(G::NamedTuple, s::CholeskySolver, dZ̄::Union{Nothing,Matrix{Float64}},
                   λ̄::Union{Nothing,Matrix{Float64}})
    info = zeros(Int32, batchsize(s))
    g(x) = x === nothing ? C_NULL : pointer(x)
    GC.@preserve G s dZ̄ λ̄ info begin
        rc = ccall((:lqrb_kkt_grad_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32, Int32,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            s.handle.ptr, s.n, s.m, s.N, batchsize(s), s.p, s.hess_mode, Int32(0),
            s.Q, s.R, ptr_or_null(s.Hux), s.A, s.B, ptr_or_null(s.D2), s.C,
            s.δZ, s.λ, g(dZ̄), g(λ̄),
            g(G.Q), g(G.R), g(G.Hux), g(G.q), g(G.r), g(G.A), g(G.B), g(G.d), g(G.D2), g(G.C), g(G.c), info)
    end
    check(s.handle, rc)
    return info
end

"_solve!(solver): src/cholesky_solver.jl:166-182 — the five steps in ONE fused kernel launch"
_solve!(s::CholeskySolver) = (s.Ginv = true; _call_kkt!(s, Int32(0)))
"second_order_correction!: src/cholesky_solver.jl:254-273 (the Ginv=false chain)"
second_order_correction!(s::CholeskySolver) = (s.Ginv = false; _call_kkt!(s, FLAG_SOC))

# ---- the five steps one by one (test/cholesky_solve.jl:14-35): two launches on the general kernel
"calculate_shur_factors!(F, Jinv, blocks[, Ginv]): src/jacobian_blocks.jl:220-229.  On the device S is formed block
row by block row inside the factor launch (cholesky! below); this call fixes Ginv."
function calculate_shur_factors!(F::ShurBlocks, Jinv=nothing, blocks=nothing, Ginv::Bool=true)
    F.solver.Ginv = Ginv
    F.solver.factored = false
    return F
end
"cholesky!(U, F): src/cholesky_solve.jl:28-33 = lqrb_kkt_factor_f64; the handle keeps the block rows of U"
function LinearAlgebra.cholesky!(U::ShurBlocks, F::ShurBlocks)
    s = U.solver
    GC.@preserve s begin
        rc = ccall((:lqrb_kkt_factor_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32, Int32,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            s.handle.ptr, s.n, s.m, s.N, batchsize(s), s.p, s.hess_mode, _flags(s),
            s.Q, s.R, ptr_or_null(s.Hux), s.A, s.B, ptr_or_null(s.D2), s.C, s.info)
    end
    check(s.handle, rc)
    s.factored = true
    return U
end
"solve with the kept factor and a right-hand side (default: the solver's own q, r, d, c): lqrb_kkt_solve_factored_f64"
function solve_factored!(s::CholeskySolver; q=s.q, r=s.r, d=s.d, c=s.c)
    s.factored || cholesky!(s.chol_blocks, s.shur_blocks)
    GC.@preserve s q r d c begin
        rc = ccall((:lqrb_kkt_solve_factored_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32, Int32, Int32,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            s.handle.ptr, s.n, s.m, s.N, batchsize(s), s.p, s.hess_mode, Int32(s.D2 !== nothing), _flags(s),
            q, r, d, c, s.δZ, s.λ, s.res, s.info)
    end
    check(s.handle, rc)
    return s
end
"forward_substitution!(chol): src/cholesky_solve.jl:93-117 — first half of the solve_factored! launch"
forward_substitution!(U::ShurBlocks) = (solve_factored!(U.solver); U)
"backward_substitution!(chol): src/cholesky_solve.jl:119-143 — second half of the same launch (already done)"
backward_substitution!(U::ShurBlocks) = U
"calculate_primals!(δZ, Jinv, chol, blocks): src/cholesky_solver.jl:185-199"
calculate_primals!(δZ, Jinv, U::ShurBlocks, blocks=nothing) = (δZ .= U.solver.δZ; δZ)

function _dense_factors(s::CholeskySolver)
    P, b = size(s.λ, 1), batchsize(s)
    S, U, h = zeros(P, P, b), zeros(P, P, b), zeros(P, b)
    GC.@preserve s S U h begin
        rc = ccall((:lqrb_kkt_get_shur_f64, lib), Int32,
            (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32, Int32,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
            s.handle.ptr, s.n, s.m, s.N, b, s.p, s.hess_mode, _flags(s),
            s.Q, s.R, ptr_or_null(s.Hux), s.q, s.r, s.A, s.B, s.d, ptr_or_null(s.D2), s.C, s.c,
            S, h, U, Ptr{Int32}(C_NULL))
    end
    check(s.handle, rc)
    return S, h, U
end
"get_shur_factors(solver): (S, h, λ) per instance, src/cholesky_solver.jl:333-341"
get_shur_factors(s::CholeskySolver) = ((S, h, _) = _dense_factors(s); (S, h, s.λ))
"get_cholesky(solver): dense upper-triangular U, U'U = S, src/cholesky_solver.jl:352-359"
get_cholesky(s::CholeskySolver) = _dense_factors(s)[3]
"copy_shur_factors!(S, h, λ, F): src/jacobian_blocks.jl:173-180 on the device's block rows"
function copy_shur_factors!(S, h, λ, F::ShurBlocks)
    Sd, hd, Ud = _dense_factors(F.solver)
    S .= (F.kind == :shur ? Sd : Ud)
    h .= hd
    λ .= F.solver.λ
    return S, h, λ
end

"residual(solver; recalculate): src/cholesky_solver.jl:238-252.  recalculate=true evaluates res on the device from
the solver's current blocks and the multipliers kept from the last solve (calc_residual!, :201-236)."
function residual(s::CholeskySolver; recalculate::Bool=false)
    n, m, N = size(s)
    if recalculate
        s.linearize! === nothing || s.linearize!(s)
        norms = zeros(batchsize(s))
        GC.@preserve s norms begin
            rc = ccall((:lqrb_kkt_residual_f64, lib), Int32,
                (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32,
                 Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                 Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                s.handle.ptr, s.n, s.m, s.N, batchsize(s), s.p, _flags(s),
                s.q, s.r, s.A, s.B, ptr_or_null(s.D2), s.C, s.λ, s.res, norms)
        end
        check(s.handle, rc)
        return norms
    end
    map(1:batchsize(s)) do i
        r = view(s.res, :, i)
        norm([norm(view(r, (k - 1) * (n + m) .+ (1:(k < N ? n + m : n)))) for k = 1:N])
    end
end
get_step(s::CholeskySolver) = s.δZ
get_multipliers(s::CholeskySolver) = s.λ
get_residual(s::CholeskySolver) = s.res

"update!(solver): src/cholesky_solver.jl:155-164 — the caller's linearisation fills the blocks from solver.Z"
update!(s::CholeskySolver) = (s.linearize! === nothing || s.linearize!(s); s.factored = false; s)

"step!(solver): src/cholesky_solver.jl:122-153 with full steps (the reference's line search is TrajectoryOptimization's;
the on-device globalised loop for the Dubins car is solve!(::DubinsSQP) below).  Returns true when every instance
has feas_p, feas_d < 1e-5."
function step!(s::CholeskySolver; ϵ_p=1e-5, ϵ_d=1e-5)
    update!(s)
    feas_d = residual(s, recalculate=false)
    feas_p = s.max_violation === nothing ? fill(Inf, batchsize(s)) : s.max_violation(s)
    all(feas_p .< ϵ_p) && all(feas_d .< ϵ_d) && return true
    _solve!(s)
    s.Z .+= s.δZ
    return false
end
"solve!(solver): src/cholesky_solver.jl:109-120 — at most 10 outer iterations"
function solve!(s::CholeskySolver; iters::Int=10)
    update!(s)
    for i = 1:iters
        step!(s) && break
    end
    return s
end

# ------------------------------------------------------------------ Dubins SQP on the device (config 4) ---
struct SqpOptions
    N::Int32
    iters::Int32
    dt::Float64
    q_diag::Float64
    r_diag::Float64
    qf_diag::Float64
    eps_p::Float64
    eps_d::Float64
    line_search::Int32
end
"solve!/step! (src/cholesky_solver.jl:109-153) globalised as src/sqp.jl:72-94, entirely on the device: RK3
linearisation, cost expansion, one constrained KKT solve per iteration, L1 merit + back-tracking + SOC."
mutable struct DubinsSQP
    handle::Handle
    opts::SqpOptions
    x0::Matrix{Float64}   # 3×batch
    xf::Matrix{Float64}
    feas_p::Vector{Float64}
    feas_d::Vector{Float64}
    iters::Vector{Int32}
    kkt_solves::Int64
end
function DubinsSQP(handle::Handle, x0::Matrix{Float64}, xf::Matrix{Float64}; N=101, tf=3.0, iters=10, Q=1e-2, R=1e-2, Qf=100.0,
                   line_search=true)
    b = size(x0, 2)
    DubinsSQP(handle, SqpOptions(N, iters, tf / (N - 1), Q, R, Qf, 1e-5, 1e-5, line_search ? 1 : 0), x0, xf,
              zeros(b), zeros(b), zeros(Int32, b), 0)
end
"solve!(solver::DubinsSQP, Z): Z (NN×batch, Primals order) is the initial guess on entry and the solution on exit"
function solve!(s::DubinsSQP, Z::Matrix{Float64})
    solves = Ref{Int64}(0)
    opts = Ref(s.opts)
    GC.@preserve s Z begin
        rc = ccall((:lqrb_sqp_dubins_f64, lib), Int32,
            (Ptr{Cvoid}, Int64, Ref{SqpOptions}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Int32}, Ref{Int64}),
            s.handle.ptr, size(Z, 2), opts, s.x0, s.xf, Z, s.feas_p, s.feas_d, s.iters, solves)
    end
    check(s.handle, rc)
    s.kkt_solves = solves[]
    return Z
end

# ------------------------------------------------------------------ device-resident split (raw device pointers)
# For callers that keep their data on the GPU (e.g. through CUDA.jl's `pointer(::CuArray)`): pack once, solve
# many times without host copies, unpack.  Sizes come from riccati_layout / kkt_data_rows / padded_batch.
riccati_pack!(h::Handle, n, m, N, batch, flags, A::DevPtr, B::DevPtr, Q::DevPtr, R::DevPtr, q::DevPtr, r::DevPtr, Qf::DevPtr,
              qf::DevPtr, x0::DevPtr, knots::DevPtr, term::DevPtr) =
    check(h, ccall((:lqrb_riccati_pack_f64, lib), Int32,
        (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        h.ptr, n, m, N, batch, flags, A, B, Q, R, q, r, Qf, qf, x0, knots, term))
riccati_solve_packed!(h::Handle, n, m, N, batch, flags, knots::DevPtr, term::DevPtr, Z::DevPtr, gains::DevPtr, info::Ptr{Int32}) =
    check(h, ccall((:lqrb_riccati_solve_packed_f64, lib), Int32,
        (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
        h.ptr, n, m, N, batch, flags, knots, term, Z, gains, info))
riccati_unpack!(h::Handle, n, m, N, batch, Zp::DevPtr, gains::DevPtr, Z::DevPtr, K::DevPtr, kff::DevPtr) =
    check(h, ccall((:lqrb_riccati_unpack_f64, lib), Int32,
        (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        h.ptr, n, m, N, batch, Zp, gains, Z, K, kff))
unpack_rows!(h::Handle, rows, batch, tile, packed::DevPtr, out::DevPtr) =
    check(h, ccall((:lqrb_unpack_rows_f64, lib), Int32, (Ptr{Cvoid}, Int64, Int64, Int32, Ptr{Float64}, Ptr{Float64}),
        h.ptr, rows, batch, tile, packed, out))
pack_rows!(h::Handle, rows, batch, tile, src::DevPtr, packed::DevPtr) =
    check(h, ccall((:lqrb_pack_rows_f64, lib), Int32, (Ptr{Cvoid}, Int64, Int64, Int32, Ptr{Float64}, Ptr{Float64}),
        h.ptr, rows, batch, tile, src, packed))
kkt_pack!(h::Handle, n, m, N, batch, p::Vector{Int32}, hess_mode, Q::DevPtr, R::DevPtr, Hux::DevPtr, q::DevPtr, r::DevPtr, A::DevPtr,
          B::DevPtr, d::DevPtr, D2::DevPtr, C::DevPtr, c::DevPtr, data::DevPtr) =
    check(h, ccall((:lqrb_kkt_pack_f64, lib), Int32,
        (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        h.ptr, n, m, N, batch, p, hess_mode, Q, R, Hux, q, r, A, B, d, D2, C, c, data))
kkt_solve_packed!(h::Handle, n, m, N, batch, p::Vector{Int32}, hess_mode, explicit_d2, flags, data::DevPtr, dz::DevPtr, mult::DevPtr,
                  res::DevPtr, info::Ptr{Int32}) =
    check(h, ccall((:lqrb_kkt_solve_packed_f64, lib), Int32,
        (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Int32}),
        h.ptr, n, m, N, batch, p, hess_mode, explicit_d2, flags, data, dz, mult, res, info))
kkt_unpack!(h::Handle, n, m, N, batch, p::Vector{Int32}, hess_mode, explicit_d2, dzp::DevPtr, multp::DevPtr, resp::DevPtr, dz::DevPtr,
            mult::DevPtr, res::DevPtr) =
    check(h, ccall((:lqrb_kkt_unpack_f64, lib), Int32,
        (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Int32}, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}),
        h.ptr, n, m, N, batch, p, hess_mode, explicit_d2, dzp, multp, resp, dz, mult, res))

export Handle, LQRBError, LQRProblem, LQRSolution, DPSolver, LeastSquaresSolver, solve!, rollout!, riccati_grad!, riccati_grad_gains!, dare!, dare_grad!, admm_cache!, admm_solve!, kkt_grad!, num_vars,
       state, control,
       BlockCholesky, InvertedQuadratic, update_cost!, update_cholesky!, gradient,
       ConstraintBlock, ConstraintBlocks, dims, copy_blocks!, gen_con_inds,
       CholeskySolver, build_shur_factors, calculate_shur_factors!, forward_substitution!, backward_substitution!,
       calculate_primals!, solve_factored!, copy_shur_factors!, get_shur_factors, get_cholesky,
       _solve!, step!, update!, second_order_correction!, residual, get_step, get_multipliers, get_residual,
       DubinsSQP, SqpOptions, riccati_pack!, riccati_solve_packed!, riccati_unpack!, kkt_pack!, kkt_solve_packed!,
       kkt_unpack!, pack_rows!, unpack_rows!, riccati_layout, kkt_data_rows, kkt_knot_offset, padded_batch, num_cons,
       riccati_tile_width, kkt_tile_width, set_stream!, set_option!, synchronize, launch_count, last_kernel_name,
       fp64_peak, version, device_count, kkt_last_condition

end # module
