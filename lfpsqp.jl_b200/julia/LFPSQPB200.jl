# LFPSQPB200.jl -- thin `ccall` layer over liblfpsqp_b200.so (include/lfpsqp_b200.h) keeping LFPSQP.jl's
# `optimize(...)` method family and its `(x, obj_values, λ_kkt, term_info)` return (src/optimize.jl:13-114, :442).
#
# NOTE: Julia is not installed in the build image, so this file has never been executed; the identical call sequence
# is exercised through the ctypes mirror `lfpsqp.jl_b200/api.py`.  No CUDA.jl, no array dispatch: plain pointers.
module LFPSQPB200
import Random

export optimize, optimize_batched, optimize_large, LFPSQPParams, TerminationInfo, DeviceFamily, DeviceCallback, callbacks, use_devices!,
       rosenbrock, readme_equality,
       readme_inequality, thomson, diagquad, qcqp, QCQPFamily

const lib = joinpath(@__DIR__, "..", "liblfpsqp_b200.so")

@enum TerminationCondition f_tol x_tol kkt_tol max_iter armijo_error   # src/LFPSQP.jl:37-43

# lfpsqp_params == LFPSQPParams (src/LFPSQP.jl:57-81), C layout
Base.@kwdef struct LFPSQPParams
    α::Float64 = 1.0;  β::Float64 = 0.0;  t_β::Int64 = 0;  s::Float64 = 0.5;  σ::Float64 = 1e-4
    ϵ_c::Float64 = 1e-6;  ϵ_f::Float64 = 1e-6;  ϵ_x::Float64 = 0.0;  ϵ_kkt::Float64 = 1e-6;  ϵ_rank::Float64 = 1e-10
    maxiter::Int64 = 10000;  maxiter_retract::Int64 = 100;  maxiter_pcg::Int64 = 100;  μ0::Float64 = 1e-2
    disable_linesearch::Int32 = 0;  do_project_retract::Int32 = 1;  disp::Int32 = 1;  linesearch::Int32 = 0
    do_newton::Int32 = 1;  _pad::Int32 = 0;  tn_maxiter::Int64 = 10000;  tn_κ::Float64 = 0.5;  callback_period::Int64 = 100
end

struct CTerm                      # lfpsqp_term (TerminationInfo + status bits in the enum's padding)
    condition::Int32; status::Int32; f_diff::Float64; step_diff::Float64; kkt_diff::Float64; iter::Int64
end

struct TerminationInfo            # src/LFPSQP.jl:45-51
    condition::TerminationCondition; f_diff::Float64; step_diff::Float64; kkt_diff::Float64; iter::Int64
end

# registered device family: id + parameter blob (replaces the closures f, c!, d!)
struct DeviceFamily
    id::Cint; n::Int64; m::Int64; p::Int64; params::Vector{Float64}; stride::Int64
end
rosenbrock() = DeviceFamily(0, 2, 0, 0, Float64[], 0)
readme_equality(n=50) = DeviceFamily(1, n, 1, 0, Float64[], 0)
readme_inequality(coeff::Vector{Float64}) = DeviceFamily(2, length(coeff), 0, 1, coeff, 0)
readme_inequality(coeff::Matrix{Float64}) = DeviceFamily(2, size(coeff, 1), 0, 1, vec(coeff), size(coeff, 1))  # n x B
thomson(N) = DeviceFamily(3, 3N, N, 0, Float64[], 0)
diagquad(Q, A, b, xt, w) = DeviceFamily(4, size(Q, 2), size(Q, 1), 0,
                                        vcat(vec(permutedims(Q)), vec(permutedims(A)), b, xt, w), 0)  # row-major Q, A

const ctx = Ref{Ptr{Cvoid}}(C_NULL)
function context()
    if ctx[] == C_NULL
        rc = ccall((:lfpsqp_ctx_create, lib), Cint, (Cint, Ptr{Ptr{Cvoid}}), 0, ctx)
        rc == 0 || error(unsafe_string(ccall((:lfpsqp_last_error, lib), Cstring, (Ptr{Cvoid},), C_NULL)))
    end
    ctx[]
end
check(rc) = rc == 0 || error(unsafe_string(ccall((:lfpsqp_last_error, lib), Cstring, (Ptr{Cvoid},), ctx[])))

"B independent instances: X0 is n x B (column-major, one instance per column)."
function optimize_batched(fam::DeviceFamily, X0::Matrix{Float64}, xl, xu, param::LFPSQPParams=LFPSQPParams(); history::Int=64)
    n, B = size(X0); me = fam.m + fam.p
    x = Matrix{Float64}(undef, n, B); obj = Matrix{Float64}(undef, history, B); len = Vector{Int64}(undef, B)
    λ = Matrix{Float64}(undef, me, B); term = Vector{CTerm}(undef, B)
    pl = isnothing(xl) ? Ptr{Float64}(C_NULL) : pointer(xl); pu = isnothing(xu) ? Ptr{Float64}(C_NULL) : pointer(xu)
    GC.@preserve X0 xl xu x obj len λ term fam begin
        check(ccall((:lfpsqp_solve_batched, lib), Cint,
                    (Ptr{Cvoid}, Cint, Int64, Int64, Int64, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64},
                     Ptr{Float64}, Ref{LFPSQPParams}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Float64},
                     Ptr{CTerm}, Ptr{Cvoid}),
                    context(), fam.id, n, fam.m, fam.p, B, fam.params, fam.stride, X0, pl, pu, param, x, obj, history,
                    len, λ, term, C_NULL))
    end
    x, obj, len, λ, term
end

# dense QCQP given by data (LFPSQP_FAM_QCQP = 101): lfpsqp_qcqp is nine {pointer, batch stride} pairs
struct CQcqp
    P::Ptr{Float64}; P_stride::Int64; q::Ptr{Float64}; q_stride::Int64; r::Ptr{Float64}; r_stride::Int64
    Qc::Ptr{Float64}; Qc_stride::Int64; Ac::Ptr{Float64}; Ac_stride::Int64; bc::Ptr{Float64}; bc_stride::Int64
    Qd::Ptr{Float64}; Qd_stride::Int64; Ad::Ptr{Float64}; Ad_stride::Int64; bd::Ptr{Float64}; bd_stride::Int64
end
struct QCQPFamily
    n::Int64; m::Int64; p::Int64; arrays::Vector{Any}; strides::Vector{Int64}   # P q r Qc Ac bc Qd Ad bd (nothing = zero)
end
const _QCQP_NDIMS = (2, 1, 0, 3, 2, 1, 3, 2, 1)   # own dims: P n x n, q n, r scalar, Qc n x n x m, Ac n x m (column i = a_i), bc m, ...
"""qcqp(; P, q, r, Qc, Ac, bc, Qd, Ad, bd): each array at its own shape (shared by the batch) or with a trailing batch
dimension B (per instance); nothing = zero.  Matrices are symmetrised as (M + M')/2."""
function qcqp(; P=nothing, q=nothing, r=nothing, Qc=nothing, Ac=nothing, bc=nothing, Qd=nothing, Ad=nothing, bd=nothing)
    arrays = Any[P, q, r, Qc, Ac, bc, Qd, Ad, bd]; strides = zeros(Int64, 9)
    for i in 1:9
        a = arrays[i]
        isnothing(a) && continue
        a = Array{Float64}(a isa Number ? fill(Float64(a)) : a)
        if i in (1, 4, 7)   # symmetrise every n x n slice
            a = (a .+ permutedims(a, (2, 1, (3:ndims(a))...))) ./ 2
        end
        ndims(a) == _QCQP_NDIMS[i] + 1 && (strides[i] = prod(size(a)[1:end-1]))
        ndims(a) in (_QCQP_NDIMS[i], _QCQP_NDIMS[i] + 1) || error("qcqp: array $i has $(ndims(a)) dimensions")
        arrays[i] = a
    end
    n = something(map(a -> isnothing(a) ? nothing : size(a, 1), arrays[[1, 2, 4, 5, 7, 8]])..., 0)
    m = isnothing(bc) ? (isnothing(Ac) ? (isnothing(Qc) ? 0 : size(arrays[4], 3)) : size(arrays[5], 2)) : size(arrays[6], 1)
    p = isnothing(bd) ? (isnothing(Ad) ? (isnothing(Qd) ? 0 : size(arrays[7], 3)) : size(arrays[8], 2)) : size(arrays[9], 1)
    QCQPFamily(n, m, p, arrays, strides)
end

function optimize_batched(fam::QCQPFamily, X0::Matrix{Float64}, xl, xu, param::LFPSQPParams=LFPSQPParams(); history::Int=64)
    n, B = size(X0); me = fam.m + fam.p
    x = Matrix{Float64}(undef, n, B); obj = Matrix{Float64}(undef, history, B); len = Vector{Int64}(undef, B)
    λ = Matrix{Float64}(undef, me, B); term = Vector{CTerm}(undef, B)
    pl = isnothing(xl) ? Ptr{Float64}(C_NULL) : pointer(xl); pu = isnothing(xu) ? Ptr{Float64}(C_NULL) : pointer(xu)
    GC.@preserve X0 xl xu x obj len λ term fam begin
        ptrs = [isnothing(a) ? Ptr{Float64}(C_NULL) : pointer(a) for a in fam.arrays]
        desc = Ref(CQcqp(collect(Iterators.flatten(zip(ptrs, fam.strides)))...))
        check(ccall((:lfpsqp_solve_batched, lib), Cint,
                    (Ptr{Cvoid}, Cint, Int64, Int64, Int64, Int64, Ref{CQcqp}, Int64, Ptr{Float64}, Ptr{Float64},
                     Ptr{Float64}, Ref{LFPSQPParams}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Float64},
                     Ptr{CTerm}, Ptr{Cvoid}),
                    context(), 101, n, fam.m, fam.p, B, desc, 0, X0, pl, pu, param, x, obj, history,
                    len, λ, term, C_NULL))
    end
    x, obj, len, λ, term
end

# optimize(f, c!, d!, x0, xl, xu, m, p[, param])  (src/optimize.jl:83) -- f, c!, d! are replaced by the family handle
function optimize(fam::DeviceFamily, x0::Vector{Float64}, xl, xu, param::LFPSQPParams=LFPSQPParams())
    x, obj, len, λ, term = optimize_batched(fam, reshape(x0, :, 1), xl, xu, param; history=param.maxiter + 1)
    t = term[1]
    t.iter == param.maxiter && @warn "Maximum # of outer iterations reached"          # optimize.jl:438-440
    x[:, 1], obj[1:len[1], 1], λ[:, 1], TerminationInfo(TerminationCondition(t.condition), t.f_diff, t.step_diff, t.kkt_diff, t.iter)
end
optimize(fam::DeviceFamily, x0::Vector{Float64}, param::LFPSQPParams=LFPSQPParams()) = optimize(fam, x0, nothing, nothing, param)

# ---------------------------------------------------------------------------------------------------------------
# The reference's own method family (src/optimize.jl:13, :83, :88, :107, :112) with DEVICE-CALLBACK HANDLES in the
# positions of the closures f, c!, d!: `cb = callbacks(fam)` gives `cb.f`, `cb.c!`, `cb.d!` (nothing when the family has
# no such role), and then
#     x, obj_values, λ_kkt, term_info = optimize(cb.f, cb.c!, cb.d!, x0, xl, xu, m, p)          # the north-star shape
# is the call a user of LFPSQP.jl writes today, argument for argument (same order, same `nothing` conventions, same
# error() conditions, same 4-tuple with the untruncated λ of length m+p, optimize.jl:67-70).  lfpsqp.jl_b200/api.py is
# the executed mirror of exactly these methods.
struct DeviceCallback
    family::DeviceFamily
    role::Symbol                  # :f, :c, :d
end
callbacks(fam::DeviceFamily) = (f = DeviceCallback(fam, :f), c! = fam.m > 0 ? DeviceCallback(fam, :c) : nothing,
                                d! = fam.p > 0 ? DeviceCallback(fam, :d) : nothing)
function _family(f::DeviceCallback, c!, d!)
    f.role == :f || error("f must be the f handle of a registered device family")
    for (cb, role) in ((c!, :c), (d!, :d))
        isnothing(cb) && continue
        (cb isa DeviceCallback && cb.family === f.family && cb.role == role) || error("$(role)! must be the $(role) handle of the same family as f")
    end
    f.family
end
function _solve(fam::DeviceFamily, x0, xl, xu, m, p, param)
    (length(x0), m, p) == (fam.n, fam.m, fam.p) || error("sizes (n=$(length(x0)), m=$m, p=$p) do not match the family")
    optimize(fam, x0, xl, xu, param)
end
# optimize(f, c!, d!, dl, du, x0, xl, xu, m, p[, param])                                             (optimize.jl:13)
function optimize(f::DeviceCallback, c!, d!, dl, du, x0::Vector{Float64}, xl, xu, m::Int64, p::Int64, param::LFPSQPParams=LFPSQPParams())
    fam = _family(f, c!, d!)
    if isnothing(d!) || p == 0                                                                        # optimize.jl:15-17
        return optimize(f, c!, x0, xl, xu, m, param)
    end
    (length(dl) == length(du) == p) || error("Bound vectors dl and du must be of size p")             # optimize.jl:19-21
    (all(==(-Inf), dl) && all(==(0.0), du)) || error("only d(x) <= 0 (dl = -Inf, du = 0; optimize.jl:83-85) is on the device path")
    n = length(x0)
    _solve(fam, x0, isnothing(xl) ? fill(-Inf, n) : xl, isnothing(xu) ? fill(Inf, n) : xu, m, p, param)   # optimize.jl:30-36
end
# optimize(f, c!, d!, x0, xl, xu, m, p[, param])                                                     (optimize.jl:83-85)
optimize(f::DeviceCallback, c!, d!, x0::Vector{Float64}, xl, xu, m::Int64, p::Int64, param::LFPSQPParams=LFPSQPParams()) =
    optimize(f, c!, d!, fill(-Inf, p), zeros(p), x0, xl, xu, m, p, param)
# optimize(f, c!, x0, xl, xu, m[, param])                                                            (optimize.jl:88-104)
function optimize(f::DeviceCallback, c!, x0::Vector{Float64}, xl, xu, m::Int64, param::LFPSQPParams=LFPSQPParams())
    fam = _family(f, c!, nothing)
    if !isnothing(xl) && !isnothing(xu) && !(length(xl) == length(xu) == length(x0))
        error("xl, xu, and x0 must all be the same length")                                           # optimize.jl:144-148
    end
    isnothing(xl) == isnothing(xu) || error("xl and xu must both be given or both be nothing")
    _solve(fam, x0, xl, xu, m, 0, param)
end
# optimize(f, c!, x0, m[, param]) and optimize(f, x0[, param])                                        (optimize.jl:107-114)
optimize(f::DeviceCallback, c!, x0::Vector{Float64}, m::Int64, param::LFPSQPParams=LFPSQPParams()) = optimize(f, c!, x0, nothing, nothing, m, param)
optimize(f::DeviceCallback, x0::Vector{Float64}, param::LFPSQPParams=LFPSQPParams()) = optimize(f, nothing, x0, nothing, nothing, 0, param)

# Multi-GPU context (lfpsqp_ctx_create_multi): every later optimize_batched call shards its instances over `devices` from one
# host call (one host thread and one stream pipeline per device inside the library, no collective).
function use_devices!(devices::Vector{<:Integer})
    ctx[] == C_NULL || ccall((:lfpsqp_ctx_destroy, lib), Cvoid, (Ptr{Cvoid},), ctx[])
    ctx[] = C_NULL
    devs = Cint.(devices)
    rc = ccall((:lfpsqp_ctx_create_multi, lib), Cint, (Ptr{Cint}, Cint, Ptr{Ptr{Cvoid}}), devs, length(devs), ctx)
    rc == 0 || error(unsafe_string(ccall((:lfpsqp_last_error, lib), Cstring, (Ptr{Cvoid},), C_NULL)))
    nothing
end


# ---------------------------------------------------------------------------------------------------------------
# Generic problems: the explicit-derivative core optimize(f, grad!, c!, jac!, hess_lag_vec!, x0, xl, xu, m, param)
# (src/optimize.jl:119-443) over lfpsqp_solve_host.  The callbacks are the reference's own closures (AD-generated by
# src/autodiff_generators.jl or hand-written); they run on the host, the linear algebra on the device.
struct HostCallbacks              # lfpsqp_host_callbacks (include/lfpsqp_b200.h)
    user::Ptr{Cvoid}; f::Ptr{Cvoid}; grad::Ptr{Cvoid}; c::Ptr{Cvoid}; jac::Ptr{Cvoid}; hess::Ptr{Cvoid}
    callback::Ptr{Cvoid}; randn::Ptr{Cvoid}
end
mutable struct HostProblem
    f; grad!; c!; jac!; hess_lag_vec!; callback; err::Any
end
_prob(u) = unsafe_pointer_to_objref(u)::HostProblem
_w(p, dims...) = unsafe_wrap(Array, p, dims)
# exceptions must not unwind through C: store them, return 1 (=> LFPSQP_ERR_CALLBACK), rethrow after the ccall
macro guarded(u, ex)
    quote
        try
            $(esc(ex)); Cint(0)
        catch e
            _prob($(esc(u))).err = e; Cint(1)
        end
    end
end
_f(u, x, n, out)::Cint = @guarded u unsafe_store!(out, _prob(u).f(_w(x, n)))
_grad(u, g, x, n)::Cint = @guarded u _prob(u).grad!(_w(g, n), _w(x, n))
_c(u, cv, x, n, m)::Cint = @guarded u _prob(u).c!(_w(cv, m), _w(x, n))
_jac(u, Jc, cv, x, n, m)::Cint = @guarded u _prob(u).jac!(_w(Jc, m, n), _w(cv, m), _w(x, n))     # Jc m x n column-major (optimize.jl:189)
_hess(u, dest, src, x, lam, n, m)::Cint = @guarded u _prob(u).hess_lag_vec!(_w(dest, n), _w(src, n), _w(x, n), _w(lam, m))
_cb(u, i, x, na)::Cint = @guarded u _prob(u).callback(i, _w(x, na))                               # optimize.jl:432-434
_randn(u, buf, na)::Cint = @guarded u Random.randn!(_w(buf, na))                                  # optimize.jl:264-273

function optimize(f, grad!, c!, jac!, hess_lag_vec!, x0::Vector{Float64}, xl, xu, m::Int64,
                  param::LFPSQPParams=LFPSQPParams(); callback=nothing)
    n = length(x0)
    if !isnothing(xl) && !isnothing(xu) && !(length(xl) == length(xu) == n)
        error("xl, xu, and x0 must all be the same length")                                       # optimize.jl:144-148
    end
    prob = HostProblem(f, grad!, c!, jac!, hess_lag_vec!, callback, nothing)
    P = Ptr{Cvoid}; D = Ptr{Float64}
    cb = HostCallbacks(pointer_from_objref(prob),
        @cfunction(_f, Cint, (P, D, Int64, D)), @cfunction(_grad, Cint, (P, D, D, Int64)),
        m > 0 ? @cfunction(_c, Cint, (P, D, D, Int64, Int64)) : C_NULL,
        m > 0 ? @cfunction(_jac, Cint, (P, D, D, D, Int64, Int64)) : C_NULL,
        @cfunction(_hess, Cint, (P, D, D, D, D, Int64, Int64)),
        isnothing(callback) ? C_NULL : @cfunction(_cb, Cint, (P, Int64, D, Int64)),
        param.β > 0 ? @cfunction(_randn, Cint, (P, D, Int64)) : C_NULL)
    H = param.maxiter + 1
    x = Vector{Float64}(undef, n); obj = Vector{Float64}(undef, H); len = Ref{Int64}(0)
    λ = Vector{Float64}(undef, max(m, 1)); term = Ref{CTerm}()
    pl = isnothing(xl) ? D(C_NULL) : pointer(xl); pu = isnothing(xu) ? D(C_NULL) : pointer(xu)
    rc = GC.@preserve prob x0 xl xu x obj λ ccall((:lfpsqp_solve_host, lib), Cint,
            (P, Ref{HostCallbacks}, Int64, Int64, D, D, D, Ref{LFPSQPParams}, D, D, Int64, Ref{Int64}, D, Ref{CTerm}, P),
            context(), cb, n, m, x0, pl, pu, param, x, obj, H, len, λ, term, C_NULL)
    isnothing(prob.err) || throw(prob.err)
    check(rc)
    t = term[]
    t.iter == param.maxiter && @warn "Maximum # of outer iterations reached"                      # optimize.jl:438-440
    x, obj[1:len[]], λ[1:m], TerminationInfo(TerminationCondition(t.condition), t.f_diff, t.step_diff, t.kkt_diff, t.iter)
end

# One large dense instance of a registered family on one GPU (large-n engine: DMMA Gram + Cholesky, streaming passes over J,
# persistent fused projcg / pcg kernels, 2n bound embedding when xl / xu are finite): lfpsqp_solve_large.
function optimize_large(fam::DeviceFamily, x0::Vector{Float64}, xl, xu, param::LFPSQPParams=LFPSQPParams())
    n = length(x0); m = fam.m
    H = param.maxiter + 1
    x = Vector{Float64}(undef, n); obj = Vector{Float64}(undef, H); len = Ref{Int64}(0)
    λ = Vector{Float64}(undef, max(m, 1)); term = Ref{CTerm}()
    D = Ptr{Float64}
    pl = isnothing(xl) ? D(C_NULL) : pointer(xl); pu = isnothing(xu) ? D(C_NULL) : pointer(xu)
    rc = GC.@preserve fam x0 xl xu x obj λ ccall((:lfpsqp_solve_large, lib), Cint,
            (Ptr{Cvoid}, Cint, Int64, Int64, D, D, D, D, Ref{LFPSQPParams}, D, D, Int64, Ref{Int64}, D, Ref{CTerm}, Ptr{Cvoid}),
            context(), fam.id, n, m, fam.params, x0, pl, pu, param, x, obj, H, len, λ, term, C_NULL)
    check(rc)
    t = term[]
    x, obj[1:len[]], λ[1:m], TerminationInfo(TerminationCondition(t.condition), t.f_diff, t.step_diff, t.kkt_diff, t.iter)
end

# Grafting into LFPSQP.jl itself is one method: every convenience method of src/optimize.jl:13-114 ends in the core at :119, so
#     LFPSQP.optimize(f, grad!, c!, jac!, hess_lag_vec!, x0::Vector{Float64}, xl, xu, m::Int64, param::LFPSQP.LFPSQPParams) =
#         LFPSQPB200.optimize(f, grad!, c!, jac!, hess_lag_vec!, x0, xl, xu, m, LFPSQPB200.LFPSQPParams(param); callback=param.callback)
# (with a field-by-field LFPSQPParams converter) sends the whole driver to the GPU while the AD generators stay untouched.

end # module
