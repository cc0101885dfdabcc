# BossB200.jl -- Julia-side binding of libboss_b200.so for BOSS.jl v0.6.1.
#
# NOT EXECUTED IN THIS REPOSITORY: the build image has no Julia.  The file is written against
# include/boss_b200.h and BOSS.jl's documented extension interfaces and is reviewed by inspection only; the same
# C ABI is exercised end to end from Python (boss.jl_b200/_lib.py, tests/).  Treat it as the integration recipe
# (INTEGRATION.md), to be run under Julia >= 1.10 before it is relied on.
#
# Design: NOTHING of BOSS.jl is overwritten.  The backend is selected by wrapping the maximizer and the fitter:
#
#     bo!(problem; acq_maximizer = B200AM(GridAM(problem, steps)), model_fitter = B200Fitter(SamplingMAP(; samples = 4096)), ...)
#
# `B200AM{A}` and `B200Fitter{F}` are NEW types, so their `maximize_acquisition` / `estimate_parameters` methods are
# new methods (Julia >= 1.10 rejects overwriting methods of another package during precompilation, and an override
# would also have replaced the stock path for kernels the device does not support).  Anything outside the
# accelerated path -- CustomKernel, a fitness that is neither LinFitness nor a B200ExprFitness, a model that is not a
# GaussianProcess / Semiparametric(…, GaussianProcess) -- falls back to the wrapped object's own BOSS.jl method.
#
#   reference function                                                          -> library entry point
#   model_posterior_slice (src/models/gaussian_process.jl:133-141)              -> boss_gp_fit / boss_gp_fit_batch
#   mean / var / mean_and_var / cov / mean_and_cov (:143-184)                   -> boss_gp_predict / boss_gp_cov
#   mean_and_var(post, X::Matrix{<:ForwardDiff.Dual})                           -> boss_gp_predict_grad
#   construct_acquisition(::ExpectedImprovement) (expected_improvement.jl:49-90)-> boss_ei_score / boss_mcei_score
#   maximize_acquisition(::GridAM)        (acquisition_maximizers/grid.jl:45-65)        -> boss_ei_score
#   maximize_acquisition(::SamplingAM)    (sampling.jl:20-57)                           -> boss_ei_score
#   maximize_acquisition(::OptimizationAM)(optimization.jl:55-118)                      -> boss_ei_maximize_multistart /
#                                                                                          boss_mcei_maximize_multistart
#   maximize_acquisition(::SampleOptAM)   (sample_opt.jl:41-52)                         -> boss_[mc]ei_score_topk + the above
#   maximize_acquisition(::SequentialBatchAM) (batch.jl:26-38)                          -> boss_gp_append
#   estimate_parameters(::SamplingMAP)    (model_fitters/sampling.jl:17-78)             -> boss_gp_loglik_batch
#   data_loglike + ForwardDiff gradient   (model_fitters/optimization.jl:41,153)        -> boss_gp_loglik_grad_batch
#     (Semiparametric: θ through ForwardDiff.jacobian of the parametric mean)             -> boss_gp_loglik_grad_batch_mean
#   acq(x::Vector{<:ForwardDiff.Dual})    (acquisition_maximizers/optimization.jl:36)   -> boss_ei_value_grad /
#                                                                                          boss_mcei_value_grad
#   estimate_parameters(::OptimizationMAP) (model_fitters/optimization.jl:75-164)        -> boss_gp_map_multistart
#   estimate_parameters(::SampleOptMAP)    (model_fitters/sample_opt.jl:37-48)          -> SamplingMAP batch + the above
module BossB200

using BOSS
using BOSS: GaussianProcess, GaussianProcessParams, Semiparametric, SemiparametricParams, ExperimentData,
            ModelPosteriorSlice, DefaultModelPosterior, BossProblem, BossOptions, AcquisitionMaximizer, ModelFitter,
            GridAM, SamplingAM, OptimizationAM, SampleOptAM, SequentialBatchAM, SamplingMAP, OptimizationMAP,
            SampleOptMAP, ExpectedImprovement,
            LinFitness, NonlinFitness, MAPParams, BIParams, Infinity, mean_getindex, best_so_far, get_params, y_dim
using KernelFunctions: SqExponentialKernel, Matern32Kernel, Matern52Kernel, ExponentialKernel, RationalQuadraticKernel
using Distances: Euclidean
using LinearAlgebra: diag, PosDefException
using Random: shuffle
using ForwardDiff
import Distributions
import Statistics: mean, var, cov
import StatsBase: mean_and_var, mean_and_cov

export B200AM, B200Fitter, B200ExprFitness, b200_posterior

const LIB = get(ENV, "BOSS_B200_LIB", joinpath(@__DIR__, "..", "boss.jl_b200", "lib", "libboss_b200.so"))

struct BossB200Error <: Exception
    code::Int
    msg::String
end
last_error() = unsafe_string(ccall((:boss_last_error, LIB), Cstring, ()))   # per calling thread
check(rc::Integer) = (rc < 0 && throw(BossB200Error(rc, last_error())); Int(rc))

"One GPU (`init(0)`) or, from a single Julia process, GPUs 0..n-1 (`init_multi(n)`): fits are replicated and the
host-pointer scoring / log-likelihood / multi-start calls are sharded inside the library (bit-identical results)."
init(device::Integer=0) = check(ccall((:boss_init, LIB), Cint, (Cint,), device))
init_multi(n::Integer) = check(ccall((:boss_init_multi, LIB), Cint, (Cint,), n))
shutdown() = ccall((:boss_shutdown, LIB), Cvoid, ())

# ---- what the device supports -----------------------------------------------------------------------------------
kernel_id(::SqExponentialKernel) = 0
kernel_id(::Matern32Kernel) = 1
kernel_id(::Matern52Kernel) = 2
# ExponentialKernel (= Matern12Kernel) and RationalQuadraticKernel: the device evaluates them on the Euclidean distance
# only; any other metric keeps the stock path.  An RQ kernel's shape α is registered once per value with the library
# (boss_kernel_rational_quadratic, host-only, thread-safe) and the id is cached here.
kernel_id(k::ExponentialKernel) = k.metric isa Euclidean ? 3 : nothing
const RQ_IDS = Dict{Float64,Cint}()
const RQ_LOCK = ReentrantLock()
function kernel_id(k::RationalQuadraticKernel)
    k.metric isa Euclidean || return nothing
    a = Float64(only(k.α))
    lock(RQ_LOCK) do
        get!(RQ_IDS, a) do
            id = Ref{Cint}(-1)
            check(ccall((:boss_kernel_rational_quadratic, LIB), Cint, (Cdouble, Ref{Cint}), a, id))
            id[]
        end
    end
end
kernel_id(k::BOSS.DiscreteKernel) = kernel_id(k.kernel)
kernel_id(k) = nothing                                  # CustomKernel etc.: not accelerated -> stock BOSS.jl path
discrete_mask(k::BOSS.DiscreteKernel) = k.dims isa Missing ? nothing : Vector{UInt8}(k.dims)
discrete_mask(k) = nothing

gp_part(m::GaussianProcess) = m
gp_part(m::Semiparametric) = m.nonparametric isa GaussianProcess ? m.nonparametric : nothing
gp_part(m) = nothing
supported(model) = (g = gp_part(model); !isnothing(g) && !isnothing(kernel_id(g.kernel)))

"A NonlinFitness drawn from the expression set the device evaluates (include/boss_b200.h, boss_mcei_score):
kind 1 affine, 2 diagonal quadratic, 3 max, 4 min.  It is also an ordinary callable, so `best_so_far` works unchanged."
struct B200ExprFitness <: BOSS.Fitness
    kind::Int
    c0::Float64
    c::Vector{Float64}
    q::Vector{Float64}
    t::Vector{Float64}
end
function (f::B200ExprFitness)(y::AbstractVector{<:Real})
    f.kind == 1 && return f.c0 + sum(f.c .* y)
    f.kind == 2 && return f.c0 + sum(f.c .* y) + sum(f.q .* (y .- f.t) .^ 2)
    live = f.c .!= 0
    vals = (f.c .* y .+ f.t)[live]
    return f.c0 + (f.kind == 3 ? maximum(vals) : minimum(vals))
end

# prior mean evaluated on the host (nothing | constant | closure), gaussian_process.jl:101-103; for a Semiparametric
# model the parametric prediction is the mean (semiparametric.jl:79-92)
eval_mean(::Nothing, X::AbstractMatrix) = nothing
eval_mean(m::Real, X::AbstractMatrix) = fill(Float64(m), size(X, 2))
eval_mean(m::Function, X::AbstractMatrix) = Float64[m(x) for x in eachcol(X)]
slice_mean(model::GaussianProcess, params, slice::Int) = mean_getindex(model.mean, slice)
slice_mean(model::Semiparametric, params, slice::Int) = (x -> model.parametric(x, params.θ)[slice])
gp_params(p::GaussianProcessParams) = (p.λ, p.α, p.σ)
gp_params(p::SemiparametricParams) = (p.λ, p.α, p.σ)
cptr(::Nothing) = C_NULL
cptr(a::AbstractArray) = pointer(a)

# ---- posterior handle: one output slice, one hyper-parameter vector (the factor cache) ------------------------------
mutable struct B200Posterior <: ModelPosteriorSlice{GaussianProcess}
    handle::Ptr{Cvoid}
    mean                         # slice mean: nothing | Real | Function
    loglik::Float64
    function B200Posterior(handle, mean, loglik)
        p = new(handle, mean, loglik)
        finalizer(q -> ccall((:boss_gp_free, LIB), Cvoid, (Ptr{Cvoid},), q.handle), p)
        return p
    end
end

"Replaces model_posterior_slice -> posterior_gp -> AbstractGPs.posterior (gaussian_process.jl:133-141,199-211)."
function fit_slice(model, params, data::ExperimentData, slice::Int)
    g = gp_part(model)
    X = Matrix{Float64}(data.X)
    m = slice_mean(model, params, slice)
    mX = eval_mean(m, X)
    δ = isnothing(mX) ? Vector{Float64}(data.Y[slice, :]) : Vector{Float64}(data.Y[slice, :]) .- mX
    λ, α, σ = gp_params(params)
    λs = Vector{Float64}(λ[:, slice])
    mask = discrete_mask(g.kernel)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    ll = Ref{Cdouble}(0.0)
    rc = GC.@preserve X δ λs mask check(ccall((:boss_gp_fit, LIB), Cint,
        (Ptr{Cdouble}, Cint, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Cdouble, Cdouble, Cint, Ptr{UInt8}, Ref{Ptr{Cvoid}}, Ref{Cdouble}),
        X, size(X, 1), size(X, 2), δ, λs, α[slice], σ[slice], kernel_id(g.kernel), cptr(mask), out, ll))
    rc == 1 && throw(PosDefException(1))        # the exception the reference path raises; SafeFunction maps it to -Inf
    return B200Posterior(out[], m, ll[])
end

"`model_posterior(problem)` on the device: a DefaultModelPosterior of B200Posterior slices (a Vector of them for BIParams)."
function b200_posterior(problem::BossProblem)
    ps = get_params(problem.params)
    one(p) = DefaultModelPosterior([fit_slice(problem.model, p, problem.data, i) for i in 1:y_dim(problem.data)])
    return ps isa AbstractVector ? one.(ps) : one(ps)
end

function mean_and_var(post::B200Posterior, X::AbstractMatrix{<:Real})
    Xs = Matrix{Float64}(X)
    M = size(Xs, 2)
    pm = eval_mean(post.mean, Xs)
    μ = Vector{Float64}(undef, M); σ2 = Vector{Float64}(undef, M); st = Vector{Int32}(undef, M)
    rc = GC.@preserve Xs pm check(ccall((:boss_gp_predict, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Int32}),
        post.handle, Xs, M, cptr(pm), μ, σ2, st))
    if rc == 2   # mirror _clip_var's DomainError (gaussian_process.jl:186-194)
        i = findfirst(!=(0), st)
        throw(DomainError(σ2[i], "The posterior GP predicted variance $(σ2[i]) but only values above -1e-8 are tolerated."))
    end
    return μ, σ2
end

# ForwardDiff through the posterior (a Dual sweep through mean / var, a custom acquisition built on b200_posterior):
# one boss_gp_predict_grad call on the values gives mu, var and their x-Jacobians (the prior mean left out); the
# partials of every column follow by the chain rule, and the slice mean is added by evaluating it on the Duals, which
# also differentiates a mean closure.  The values equal the Real method's (prior + mu in the same order).  The vector
# method below reaches this one through hcat for Dual vectors too.
dual_mean(::Nothing, X::AbstractMatrix) = nothing
dual_mean(m::Real, X::AbstractMatrix) = fill(Float64(m), size(X, 2))
dual_mean(m::Function, X::AbstractMatrix) = [m(x) for x in eachcol(X)]
function mean_and_var(post::B200Posterior, X::AbstractMatrix{D}) where {T, V, N, D<:ForwardDiff.Dual{T, V, N}}
    Xs = Matrix{Float64}(ForwardDiff.value.(X))
    d, M = size(Xs)
    μ = Vector{Float64}(undef, M); σ2 = Vector{Float64}(undef, M); st = Vector{Int32}(undef, M)
    dμ = Matrix{Float64}(undef, d, M); dσ2 = Matrix{Float64}(undef, d, M)   # one posterior: index (m*d + j)
    h = Ptr{Cvoid}[post.handle]
    rc = GC.@preserve Xs h check(ccall((:boss_gp_predict_grad, LIB), Cint,
        (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
         Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Int32}),
        h, 1, 1, Xs, M, C_NULL, C_NULL, μ, σ2, dμ, dσ2, st))
    if rc == 2   # the Real method's DomainError
        i = findfirst(!=(0), st)
        throw(DomainError(σ2[i], "The posterior GP predicted variance $(σ2[i]) but only values above -1e-8 are tolerated."))
    end
    dual(v, J, m) = ForwardDiff.Dual{T}(v, ForwardDiff.Partials(ntuple(k -> sum(J[j, m] * ForwardDiff.partials(X[j, m], k)
                                                                                  for j in 1:d), N)))
    μd = [dual(μ[m], dμ, m) for m in 1:M]
    σ2d = [dual(σ2[m], dσ2, m) for m in 1:M]
    pm = dual_mean(post.mean, X)
    return (isnothing(pm) ? μd : pm .+ μd), σ2d
end
mean_and_var(post::B200Posterior, x::AbstractVector{<:Real}) = first.(mean_and_var(post, hcat(x)))
mean(post::B200Posterior, x) = mean_and_var(post, x)[1]
var(post::B200Posterior, x) = mean_and_var(post, x)[2]

function mean_and_cov(post::B200Posterior, X::AbstractMatrix{<:Real})
    Xs = Matrix{Float64}(X)
    M = size(Xs, 2)
    pm = eval_mean(post.mean, Xs)
    μ = Vector{Float64}(undef, M); Σ = Matrix{Float64}(undef, M, M)
    rc = GC.@preserve Xs pm check(ccall((:boss_gp_cov, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), post.handle, Xs, M, cptr(pm), μ, Σ))
    rc == 2 && throw(DomainError(minimum(diag(Σ)), "The posterior GP predicted a variance below -1e-8."))
    return μ, Σ
end
cov(post::B200Posterior, X::AbstractMatrix{<:Real}) = mean_and_cov(post, X)[2]

"Incremental factor cache: one more data point, same hyper-parameters (O(n^2) instead of the reference's refit)."
function append_point!(post::B200Posterior, x::AbstractVector{<:Real}, y::Real)
    xv = Vector{Float64}(x)
    mx = eval_mean(post.mean, hcat(xv))
    δ = Float64(y) - (isnothing(mx) ? 0.0 : first(mx))
    ll = Ref{Cdouble}(0.0)
    rc = check(ccall((:boss_gp_append, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cdouble, Ref{Cdouble}), post.handle, xv, δ, ll))
    rc == 1 && throw(PosDefException(1))
    post.loglik = ll[]
    return post
end

# ---- the acquisition closure (construct_safe_acquisition, src/acquisition.jl:21-25) ----------------------------------
"Callable like the reference's `acq`: `acq(x::Vector)`, `acq(X::Matrix)` (one launch sequence for the whole batch) and
`acq(x::Vector{<:ForwardDiff.Dual})` (value + analytic x-gradient from the device, re-wrapped as a Dual)."
struct B200Acquisition
    posts::Vector{DefaultModelPosterior}      # one per BI sample (a single one for MAP params)
    handles::Vector{Ptr{Cvoid}}               # sample-major: handles[(s-1)*y_dim + i]
    ydim::Int
    fitness                                   # LinFitness | B200ExprFitness
    eps::Matrix{Float64}                      # y_dim x K draws for the Monte-Carlo EI (unused for LinFitness)
    best::Union{Nothing, Float64}
    y_max::Union{Nothing, Vector{Float64}}    # nothing <=> every constraint is Infinity (cdf == 1 exactly, utils/inf.jl)
    lb::Union{Nothing, Vector{Float64}}
    ub::Union{Nothing, Vector{Float64}}
    cons::Union{Nothing, Function}
end

ymax_vector(y_max) = all(v -> v isa Infinity || v == Inf, y_max) ? nothing : Float64[v isa Infinity ? Inf : Float64(v) for v in y_max]

function B200Acquisition(problem::BossProblem, posts)
    ei = problem.acquisition
    pv = posts isa AbstractVector ? collect(posts) : [posts]
    hs = Ptr{Cvoid}[sl.handle for p in pv for sl in p.slices]
    yd = y_dim(problem.data)
    K = length(pv) == 1 ? ei.ϵ_samples : length(pv)              # ϵ_sample_count, expected_improvement.jl:115-116
    eps = ei.fitness isa LinFitness ? zeros(yd, 0) : randn(yd, K)  # sample_ϵs, :119
    dom = problem.domain
    safe = ei.cons_safe
    return B200Acquisition(pv, hs, yd, ei.fitness, eps, best_so_far(problem, ei.fitness), ymax_vector(problem.y_max),
        safe ? Vector{Float64}(dom.bounds[1]) : nothing, safe ? Vector{Float64}(dom.bounds[2]) : nothing,
        safe ? dom.cons : nothing)
end

function prior_means(acq::B200Acquisition, Xs::Matrix{Float64})
    sl = acq.posts[1].slices                  # the prior mean does not depend on the GP hyper-parameter sample
    all(s -> isnothing(s.mean), sl) && return nothing
    pm = zeros(acq.ydim, size(Xs, 2))         # y_dim contiguous per candidate = the layout boss_ei_score expects
    for (i, s) in enumerate(sl)
        mi = eval_mean(s.mean, Xs)
        isnothing(mi) || (pm[i, :] .= mi)
    end
    return pm
end
cons_mask(acq::B200Acquisition, Xs) = isnothing(acq.cons) ? nothing : UInt8[all(acq.cons(x) .>= 0) for x in eachcol(Xs)]

"Score every column of X; returns (acq values | nothing, best value, best 1-based index) with Julia argmax semantics."
function score(acq::B200Acquisition, X::AbstractMatrix{<:Real}; want_acq::Bool=true)
    Xs = Matrix{Float64}(X)
    M = size(Xs, 2)
    pm = prior_means(acq, Xs); cm = cons_mask(acq, Xs)
    out = want_acq ? Vector{Float64}(undef, M) : nothing
    bv = Ref{Cdouble}(0.0); bi = Ref{Int64}(-1)
    best = isnothing(acq.best) ? nothing : [acq.best]
    S = length(acq.posts)
    f = acq.fitness
    rc = GC.@preserve Xs pm cm out best f begin
        if f isa LinFitness
            coefs = Vector{Float64}(f.coefs)
            GC.@preserve coefs check(ccall((:boss_ei_score, LIB), Cint,
                (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
                 Ptr{Cdouble}, Ptr{Cdouble}, Ptr{UInt8}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cdouble}, Ref{Int64}),
                acq.handles, acq.ydim, S, Xs, M, cptr(pm), coefs, cptr(best), cptr(acq.y_max), cptr(acq.lb), cptr(acq.ub),
                cptr(cm), cptr(out), C_NULL, bv, bi))
        else
            check(ccall((:boss_mcei_score, LIB), Cint,
                (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Cint, Cdouble, Ptr{Cdouble}, Ptr{Cdouble},
                 Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{UInt8},
                 Ptr{Cdouble}, Ref{Cdouble}, Ref{Int64}),
                acq.handles, acq.ydim, S, Xs, M, cptr(pm), f.kind, f.c0, f.c, f.q, f.t, acq.eps, size(acq.eps, 2),
                cptr(best), cptr(acq.y_max), cptr(acq.lb), cptr(acq.ub), cptr(cm), cptr(out), bv, bi))
        end
    end
    return out, bv[], Int(bi[]) + 1
end
"The k best columns of X: (values, 1-based indices) in descending isless order (NaN first), ties to the lower index --
`sortperm(vals; rev=true)[1:k]`, selected on the device (boss_ei_score_topk for LinFitness, boss_mcei_score_topk for
a B200ExprFitness)."
function score_topk(acq::B200Acquisition, X::AbstractMatrix{<:Real}, k::Integer)
    Xs = Matrix{Float64}(X)
    M = size(Xs, 2)
    1 <= k <= M || throw(BoundsError(1:M, k))                     # as order[1:multistart] in sample_opt.jl
    f = acq.fitness
    pm = prior_means(acq, Xs); cm = cons_mask(acq, Xs)
    best = isnothing(acq.best) ? nothing : [acq.best]
    tv = Vector{Float64}(undef, k); ti = Vector{Int64}(undef, k)
    if f isa LinFitness
        coefs = Vector{Float64}(f.coefs)
        GC.@preserve Xs pm cm best coefs check(ccall((:boss_ei_score_topk, LIB), Cint,
            (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
             Ptr{Cdouble}, Ptr{Cdouble}, Ptr{UInt8}, Int64, Ptr{Cdouble}, Ptr{Int64}),
            acq.handles, acq.ydim, length(acq.posts), Xs, M, cptr(pm), coefs, cptr(best), cptr(acq.y_max), cptr(acq.lb),
            cptr(acq.ub), cptr(cm), k, tv, ti))
    else
        GC.@preserve Xs pm cm best f check(ccall((:boss_mcei_score_topk, LIB), Cint,
            (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Cint, Cdouble, Ptr{Cdouble}, Ptr{Cdouble},
             Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{UInt8}, Int64,
             Ptr{Cdouble}, Ptr{Int64}),
            acq.handles, acq.ydim, length(acq.posts), Xs, M, cptr(pm), f.kind, f.c0, f.c, f.q, f.t, acq.eps,
            size(acq.eps, 2), cptr(best), cptr(acq.y_max), cptr(acq.lb), cptr(acq.ub), cptr(cm), k, tv, ti))
    end
    return tv, ti .+ 1
end
(acq::B200Acquisition)(X::AbstractMatrix{<:Real}) = score(acq, X)[1]
(acq::B200Acquisition)(x::AbstractVector{<:Real}) = score(acq, hcat(x))[1][1]

"Value and x-gradient of the acquisition for every column of X (LinFitness: boss_ei_value_grad; B200ExprFitness: the
chain rule through the Monte-Carlo EI, boss_mcei_value_grad; prior-mean closures enter through their ForwardDiff
Jacobian evaluated on the host)."
function value_grad(acq::B200Acquisition, X::AbstractMatrix{<:Real})
    f = acq.fitness
    Xs = Matrix{Float64}(X)
    d, M = size(Xs)
    pm = prior_means(acq, Xs); cm = cons_mask(acq, Xs)
    pmg = nothing
    if !isnothing(pm)                                     # layout: index ((m-1)*d + (j-1))*y_dim + i
        pmg = zeros(acq.ydim, d, M)
        for (i, s) in enumerate(acq.posts[1].slices), m in 1:M
            s.mean isa Function && (pmg[i, :, m] .= ForwardDiff.gradient(s.mean, Xs[:, m]))
        end
    end
    vals = Vector{Float64}(undef, M); grad = Matrix{Float64}(undef, d, M)
    best = isnothing(acq.best) ? nothing : [acq.best]
    if f isa LinFitness
        coefs = Vector{Float64}(f.coefs)
        GC.@preserve Xs pm pmg cm coefs best check(ccall((:boss_ei_value_grad, LIB), Cint,
            (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
             Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{UInt8}, Ptr{Cdouble}, Ptr{Cdouble}),
            acq.handles, acq.ydim, length(acq.posts), Xs, M, cptr(pm), cptr(pmg), coefs, cptr(best), cptr(acq.y_max),
            cptr(acq.lb), cptr(acq.ub), cptr(cm), vals, grad))
    else
        GC.@preserve Xs pm pmg cm best f check(ccall((:boss_mcei_value_grad, LIB), Cint,
            (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Cdouble, Ptr{Cdouble},
             Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
             Ptr{UInt8}, Ptr{Cdouble}, Ptr{Cdouble}),
            acq.handles, acq.ydim, length(acq.posts), Xs, M, cptr(pm), cptr(pmg), f.kind, f.c0, f.c, f.q, f.t, acq.eps,
            size(acq.eps, 2), cptr(best), cptr(acq.y_max), cptr(acq.lb), cptr(acq.ub), cptr(cm), vals, grad))
    end
    return vals, grad
end
# AutoForwardDiff (the default of OptimizationAM, acquisition_maximizers/optimization.jl:36) calls acq with Dual numbers
function (acq::B200Acquisition)(x::AbstractVector{D}) where {T, V, N, D<:ForwardDiff.Dual{T, V, N}}
    xv = ForwardDiff.value.(x)
    vals, grad = value_grad(acq, hcat(xv))
    parts = ntuple(k -> sum(grad[j, 1] * ForwardDiff.partials(x[j], k) for j in eachindex(x)), N)
    return ForwardDiff.Dual{T}(vals[1], ForwardDiff.Partials(parts))
end

# ---- acquisition maximizers -----------------------------------------------------------------------------------
"Wrap any BOSS.jl acquisition maximizer: `B200AM(GridAM(...))`."
struct B200AM{A<:AcquisitionMaximizer} <: AcquisitionMaximizer
    inner::A
end

accelerated(problem::BossProblem) = supported(problem.model) && problem.acquisition isa ExpectedImprovement &&
                                   (problem.acquisition.fitness isa LinFitness || problem.acquisition.fitness isa B200ExprFitness)

function BOSS.maximize_acquisition(am::B200AM, problem::BossProblem, options::BossOptions)
    accelerated(problem) || return BOSS.maximize_acquisition(am.inner, problem, options)      # stock path
    return maximize_b200(am.inner, problem, options, B200Acquisition(problem, b200_posterior(problem)))
end

# GridAM (grid.jl:45-65): argmax over the (shuffled) grid points, one batched call
function maximize_b200(am::GridAM, problem, options, acq)
    pts = am.shuffle ? shuffle(am.points) : am.points      # shuffle copies (grid.jl:47)
    X = reduce(hcat, pts)
    _, val, idx = score(acq, X; want_acq=false)
    return X[:, idx], val
end
# SamplingAM (sampling.jl:20-57): same rejection sampler, one batched call for all samples
function draw_samples(am::SamplingAM, problem)
    xs = [BOSS._rand_in_domain(am.x_prior, problem.domain; max_attempts=am.max_attempts) for _ in 1:am.samples]
    return BOSS._reduce_samples(xs)
end
function maximize_b200(am::SamplingAM, problem, options, acq; return_all::Bool=false)
    X = draw_samples(am, problem)
    size(X, 2) == 0 && error("SamplingAM: No samples were successfully drawn!")
    vals, val, idx = score(acq, X; want_acq=return_all)
    return return_all ? (X, vals) : (X[:, idx], val)
end
# OptimizationAM (optimization.jl:55-118): all starts advance together in the device-resident multi-start driver when
# nothing on the path is a host closure; otherwise the wrapped solver runs with the batched / Dual-aware closure
function maximize_b200(am::OptimizationAM, problem, options, acq; starts=BOSS.get_starts(am.multistart, problem.domain))
    dom = problem.domain
    f = acq.fitness
    closure_free = isnothing(dom.cons) && all(s -> !(s.mean isa Function), acq.posts[1].slices) &&
                   (f isa LinFitness || f isa B200ExprFitness) && !isnothing(acq.lb)
    if !closure_free
        cons_func = isnothing(dom.cons) ? nothing : (res, x, p) -> (res .= dom.cons(x))
        return BOSS.optimize(am, acq, cons_func, dom.bounds[1], dom.bounds[2], dom.discrete, BOSS.cons_dim(dom), starts, options)
    end
    S = Matrix{Float64}(starts)
    d, M = size(S)
    aff = nothing                                         # constant prior means as an affine map c_i + 0 . x
    if any(s -> s.mean isa Real, acq.posts[1].slices)
        aff = zeros(d + 1, acq.ydim)
        for (i, s) in enumerate(acq.posts[1].slices)
            s.mean isa Real && (aff[1, i] = s.mean)
        end
    end
    best = isnothing(acq.best) ? nothing : [acq.best]
    mask = Vector{UInt8}(dom.discrete)
    bx = Vector{Float64}(undef, d); bv = Ref{Cdouble}(0.0); bi = Ref{Int64}(-1); ev = Ref{Cint}(0)
    if f isa LinFitness
        coefs = Vector{Float64}(f.coefs)
        GC.@preserve S aff coefs best mask check(ccall((:boss_ei_maximize_multistart, LIB), Cint,
            (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Cint, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
             Ptr{Cdouble}, Ptr{Cdouble}, Ptr{UInt8}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cdouble}, Ref{Int64}, Ref{Cint}),
            acq.handles, acq.ydim, length(acq.posts), S, M, 60, 8, cptr(aff), coefs, cptr(best), cptr(acq.y_max), acq.lb,
            acq.ub, mask, C_NULL, C_NULL, bx, bv, bi, ev))
    else                                                  # B200ExprFitness: the Monte-Carlo EI with this acquisition's eps
        GC.@preserve S aff f best mask check(ccall((:boss_mcei_maximize_multistart, LIB), Cint,
            (Ptr{Ptr{Cvoid}}, Cint, Cint, Ptr{Cdouble}, Int64, Cint, Cint, Ptr{Cdouble}, Cint, Cdouble, Ptr{Cdouble},
             Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
             Ptr{UInt8}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cdouble}, Ref{Int64}, Ref{Cint}),
            acq.handles, acq.ydim, length(acq.posts), S, M, 60, 8, cptr(aff), f.kind, f.c0, f.c, f.q, f.t, acq.eps,
            size(acq.eps, 2), cptr(best), cptr(acq.y_max), acq.lb, acq.ub, mask, C_NULL, C_NULL, bx, bv, bi, ev))
    end
    bv[] == -Inf && error("All optimization runs failed!")        # optim_multistart.jl:34
    return bx, bv[]
end
# SampleOptAM (sample_opt.jl:41-52)
function maximize_b200(am::SampleOptAM, problem, options, acq)
    X = draw_samples(am.sampler, problem)
    size(X, 2) == 0 && error("SamplingAM: No samples were successfully drawn!")
    _, order = score_topk(acq, X, am.optimizer.multistart)      # the best samples in sortperm(vals; rev=true) order
    starts = X[:, order]
    return maximize_b200(am.optimizer, problem, options, acq; starts)
end
# SequentialBatchAM (batch.jl:26-38): ONE fit, then an O(n^2) factor-cache append per speculative point -- the
# reference refits the posterior (O(n^3)) for every point.  Hyper-parameters do not change between the picks.
function maximize_b200(sb::SequentialBatchAM, problem, options, acq)
    prob = deepcopy(problem)
    picks = Vector{Vector{Float64}}()
    for _ in 1:sb.batch_size
        a = B200Acquisition(prob, acq.posts)                    # new best_so_far, same (extended) handles
        x, _ = maximize_b200(sb.am isa B200AM ? sb.am.inner : sb.am, prob, options, a)
        ys = [sum(mean(p.slices[i], x) for p in acq.posts) / length(acq.posts) for i in 1:acq.ydim]   # average_mean over BI samples (batch.jl:35)
        BOSS.augment_dataset!(prob, x, ys)
        for p in acq.posts, (i, sl) in enumerate(p.slices)
            append_point!(sl, x, ys[i])
        end
        push!(picks, x)
    end
    return reduce(hcat, picks), nothing
end

# ---- model fitters ----------------------------------------------------------------------------------------------
"Wrap a BOSS.jl model fitter: `B200Fitter(SamplingMAP(; samples = 4096))`."
struct B200Fitter{F<:ModelFitter} <: ModelFitter{MAPParams}
    inner::F
end

"Batched data log-likelihood: one library call for a vector of hyper-parameter vectors (sum over output slices,
gaussian_process.jl:256-266).  Non-positive-definite samples come back as -Inf (safe_data_loglike)."
function data_loglike_batch(model, data::ExperimentData, ps::AbstractVector)
    g = gp_part(model)
    X = Matrix{Float64}(data.X)
    d, n = size(X)
    S = length(ps)
    total = zeros(S)
    mask = discrete_mask(g.kernel)
    for i in 1:y_dim(data)
        parts = gp_params.(ps)
        L = Matrix{Float64}(reduce(hcat, [p[1][:, i] for p in parts]))            # d x S
        A = Float64[p[2][i] for p in parts]; N = Float64[p[3][i] for p in parts]
        # y - m(X): shared when the mean does not depend on the sample, one column per sample for Semiparametric
        Ys = model isa Semiparametric ?
            reduce(hcat, [Vector{Float64}(data.Y[i, :]) .- eval_mean(slice_mean(model, p, i), X) for p in ps]) :
            (mX = eval_mean(slice_mean(model, ps[1], i), X); isnothing(mX) ? Vector{Float64}(data.Y[i, :]) : Vector{Float64}(data.Y[i, :]) .- mX)
        ldy = Ys isa Matrix ? n : 0
        ll = Vector{Float64}(undef, S)
        GC.@preserve X Ys L A N mask check(ccall((:boss_gp_loglik_batch, LIB), Cint,
            (Ptr{Cdouble}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{UInt8}, Int64, Ptr{Cdouble}),
            X, d, n, Ys, ldy, L, A, N, kernel_id(g.kernel), cptr(mask), S, ll))
        total .+= ll
    end
    return total
end

"The same with the gradient w.r.t. (λ, α, σ) per sample -- what ForwardDiff yields through logpdf(::FiniteGP)
(model_fitters/optimization.jl:41,153).  Returns (loglik::Vector, grads::Vector of (dλ d×y_dim, dα, dσ))."
function data_loglike_grad_batch(model::GaussianProcess, data::ExperimentData, ps::AbstractVector{<:GaussianProcessParams})
    X = Matrix{Float64}(data.X)
    d, n = size(X)
    S = length(ps); yd = y_dim(data)
    total = zeros(S)
    grads = [(zeros(d, yd), zeros(yd), zeros(yd)) for _ in 1:S]
    mask = discrete_mask(model.kernel)
    for i in 1:yd
        L = Matrix{Float64}(reduce(hcat, [p.λ[:, i] for p in ps])); A = Float64[p.α[i] for p in ps]; N = Float64[p.σ[i] for p in ps]
        mX = eval_mean(mean_getindex(model.mean, i), X)
        y = isnothing(mX) ? Vector{Float64}(data.Y[i, :]) : Vector{Float64}(data.Y[i, :]) .- mX
        ll = Vector{Float64}(undef, S); G = Matrix{Float64}(undef, d + 2, S)
        GC.@preserve X y L A N mask check(ccall((:boss_gp_loglik_grad_batch, LIB), Cint,
            (Ptr{Cdouble}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{UInt8}, Int64,
             Ptr{Cdouble}, Ptr{Cdouble}), X, d, n, y, 0, L, A, N, kernel_id(model.kernel), cptr(mask), S, ll, G))
        total .+= ll
        for s in 1:S
            grads[s][1][:, i] .= G[1:d, s]; grads[s][2][i] = G[d + 1, s]; grads[s][3][i] = G[d + 2, s]
        end
    end
    return total, grads
end

"The same for a Semiparametric model, plus the gradient w.r.t. the parametric mean's θ (DESIGN.md 2.13): per output
slice, δ = y - m(X; θ) and the n × k Jacobian J = ∂m(X; θ)/∂θ of every sample (ForwardDiff.jacobian, the layout the C
ABI takes) go to one boss_gp_loglik_grad_batch_mean call, which returns αᵀJ beside the (λ, α, σ) gradient; dθ is summed
over the slices.  Returns (loglik::Vector, grads::Vector of (dθ, dλ d×y_dim, dα, dσ)).
No Julia installation was available when this method was written: it has been reviewed, not run."
function data_loglike_grad_batch(model::Semiparametric, data::ExperimentData, ps::AbstractVector{<:SemiparametricParams})
    supported(model) || throw(ArgumentError("data_loglike_grad_batch: the nonparametric part must be a GaussianProcess " *
                                            "with an SE / Matern32 / Matern52 kernel (possibly discrete)"))
    g = gp_part(model)
    X = Matrix{Float64}(data.X)
    d, n = size(X)
    S = length(ps); yd = y_dim(data); k = length(ps[1].θ)
    total = zeros(S)
    grads = [(zeros(k), zeros(d, yd), zeros(yd), zeros(yd)) for _ in 1:S]
    mask = discrete_mask(g.kernel)
    for i in 1:yd
        L = Matrix{Float64}(reduce(hcat, [p.λ[:, i] for p in ps])); A = Float64[p.α[i] for p in ps]; N = Float64[p.σ[i] for p in ps]
        Ys = reduce(hcat, [Vector{Float64}(data.Y[i, :]) .- eval_mean(slice_mean(model, p, i), X) for p in ps])   # n x S
        Js = Array{Float64}(undef, n, k, S)
        for (s, p) in enumerate(ps)
            Js[:, :, s] .= ForwardDiff.jacobian(θ -> [model.parametric(x, θ)[i] for x in eachcol(X)], p.θ)
        end
        ll = Vector{Float64}(undef, S); G = Matrix{Float64}(undef, d + 2, S); Gm = Matrix{Float64}(undef, k, S)
        GC.@preserve X Ys Js L A N mask check(ccall((:boss_gp_loglik_grad_batch_mean, LIB), Cint,
            (Ptr{Cdouble}, Cint, Cint, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Cint, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
             Cint, Ptr{UInt8}, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}),
            X, d, n, Ys, n, Js, k, k * n, L, A, N, kernel_id(g.kernel), cptr(mask), S, ll, G, Gm))
        total .+= ll
        for s in 1:S
            grads[s][1] .+= Gm[:, s]
            grads[s][2][:, i] .= G[1:d, s]; grads[s][3][i] = G[d + 1, s]; grads[s][4][i] = G[d + 2, s]
        end
    end
    return total, grads
end

# SamplingMAP (model_fitters/sampling.jl:17-78): all prior draws, ONE batched log-likelihood, first maximum
function BOSS.estimate_parameters(f::B200Fitter{<:SamplingMAP}, problem::BossProblem, options::BossOptions; return_all::Bool=false)
    supported(problem.model) || return BOSS.estimate_parameters(f.inner, problem, options; return_all)
    model, data = problem.model, problem.data
    sampler = BOSS.params_sampler(model, data)
    prior_ll = BOSS.params_loglike(model, data)
    ps = [sampler() for _ in 1:f.inner.samples]
    lls = data_loglike_batch(model, data, ps) .+ prior_ll.(ps)
    return_all && return [MAPParams(p, l) for (p, l) in zip(ps, lls)]
    b = argmax(lls)                                           # first maximum == the reference's strict `v > best_v`
    return MAPParams(ps[b], lls[b])
end
# ---- OptimizationMAP / SampleOptMAP on the device (boss_gp_map_multistart, DESIGN.md 2.15) ---------------------------
# One prior -> (kind, p0, p1) of the C tables, or nothing for a prior the device lacks
prior_entry(p::Distributions.Dirac) = (0, Float64(p.value), 0.0)
prior_entry(p::Distributions.Normal) = (1, Float64(p.μ), Float64(p.σ))
prior_entry(p::Distributions.LogNormal) = (2, Float64(p.μ), Float64(p.σ))
prior_entry(p::Distributions.Uniform) = (3, Float64(p.a), Float64(p.b))
prior_entry(p) = nothing
# the univariate parts of a lengthscale prior (product_distribution of independent components), or nothing
prior_parts(p::Distributions.Product, d) = length(p.v) == d ? collect(p.v) : nothing
prior_parts(p::Distributions.UnivariateDistribution, d) = d == 1 ? [p] : nothing
prior_parts(p, d) = (hasproperty(p, :dists) && length(p.dists) == d) ? collect(p.dists) : nothing

"(kind (d+2) × y_dim Int32, par 2 × (d+2) × y_dim) of a GaussianProcess, or nothing when a prior does not decompose into
Dirac / Normal / LogNormal / Uniform entries."
function map_prior_tables(model::GaussianProcess, d::Int, yd::Int)
    kind = zeros(Int32, d + 2, yd); par = zeros(2, d + 2, yd)
    for i in 1:yd
        parts = prior_parts(model.lengthscale_priors[i], d)
        isnothing(parts) && return nothing
        for (j, p) in enumerate(vcat(parts, [model.amplitude_priors[i], model.noise_std_priors[i]]))
            e = prior_entry(p)
            isnothing(e) && return nothing
            kind[j, i] = e[1]; par[1, j, i] = e[2]; par[2, j, i] = e[3]
        end
    end
    return kind, par
end

"All starts of all output slices in one boss_gp_map_multistart call; start s of slice i is ps[s]'s slice-i part.
The search runs in log(raw) inside [-30, 30] (not the reference's Bijectors), every slice on its own
(optimization.jl:76-84).  Returns the combined best params and their model log-likelihood (return_all: per start s)."
function map_multistart(model::GaussianProcess, data::ExperimentData, tables, ps, iters::Int; return_all::Bool=false)
    kind, par = tables
    X = Matrix{Float64}(data.X)
    d, n = size(X)
    yd = y_dim(data); M = length(ps); P = d + 2
    Y = Matrix{Float64}(undef, n, yd)
    for i in 1:yd
        mX = eval_mean(mean_getindex(model.mean, i), X)
        Y[:, i] .= isnothing(mX) ? data.Y[i, :] : data.Y[i, :] .- mX
    end
    S = Array{Float64}(undef, P, M, yd)                   # C layout [y_dim][M][P]
    for (s, p) in enumerate(ps), i in 1:yd
        S[1:d, s, i] .= p.λ[:, i]; S[d + 1, s, i] = p.α[i]; S[d + 2, s, i] = p.σ[i]
    end
    mask = discrete_mask(model.kernel)
    po = Array{Float64}(undef, P, M, yd); fo = Matrix{Float64}(undef, M, yd); bp = Matrix{Float64}(undef, P, yd)
    bv = Vector{Float64}(undef, yd); bi = Vector{Int64}(undef, yd); ev = Ref{Cint}(0)
    GC.@preserve X Y kind par S mask po fo bp bv bi check(ccall((:boss_gp_map_multistart, LIB), Cint,
        (Ptr{Cdouble}, Cint, Cint, Cint, Ptr{Cdouble}, Cint, Ptr{UInt8}, Ptr{Int32}, Ptr{Cdouble}, Ptr{Cdouble}, Int64, Cint,
         Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Int64}, Ref{Cint}),
        X, d, n, yd, Y, kernel_id(model.kernel), cptr(mask), kind, par, S, M, iters, 8, po, fo, bp, bv, bi, ev))
    any(<(0), bi) && error("All optimization runs failed!")              # optim_multistart.jl:34
    mk(rows) = GaussianProcessParams(rows[1:d, :], rows[d + 1, :], rows[d + 2, :])
    if return_all
        tot = vec(sum(fo; dims=2))
        return [MAPParams(mk(po[:, s, :]), tot[s]) for s in 1:M if isfinite(tot[s])]
    end
    return MAPParams(mk(bp), sum(bv))
end

map_tables(problem) = problem.model isa GaussianProcess && supported(problem.model) ?
    map_prior_tables(problem.model, size(problem.data.X, 1), y_dim(problem.data)) : nothing

# OptimizationMAP (optimization.jl:75-164): starts from the model's params_sampler as optimization.jl:116,131-141 draws
# them; models or priors the device lacks run the stock method.  Reviewed, not run (no Julia installation was available).
function BOSS.estimate_parameters(f::B200Fitter{<:OptimizationMAP}, problem::BossProblem, options::BossOptions;
                                  return_all::Bool=false)
    tables = map_tables(problem)
    isnothing(tables) && return BOSS.estimate_parameters(f.inner, problem, options; return_all)
    sampler = BOSS.params_sampler(problem.model, problem.data)
    ps = [sampler() for _ in 1:f.inner.multistart]
    iters = get(f.inner.kwargs, :iterations, 40)
    return map_multistart(problem.model, problem.data, tables, ps, iters; return_all)
end
# SampleOptMAP (sample_opt.jl:37-48): the SamplingMAP batch on the device, its `multistart` best samples as the starts
function BOSS.estimate_parameters(f::B200Fitter{<:SampleOptMAP}, problem::BossProblem, options::BossOptions;
                                  return_all::Bool=false)
    tables = map_tables(problem)
    isnothing(tables) && return BOSS.estimate_parameters(f.inner, problem, options; return_all)
    all_ = BOSS.estimate_parameters(B200Fitter(f.inner.sampler), problem, options; return_all=true)
    order = sortperm([p.loglike for p in all_]; rev=true)[1:f.inner.optimizer.multistart]
    ps = [all_[k].params for k in order]
    iters = get(f.inner.optimizer.kwargs, :iterations, 40)
    return map_multistart(problem.model, problem.data, tables, ps, iters; return_all)
end
# every other fitter runs its own BOSS.jl method (the accelerated batch API above is available to custom fitters)
BOSS.estimate_parameters(f::B200Fitter, problem::BossProblem, options::BossOptions; kwargs...) =
    BOSS.estimate_parameters(f.inner, problem, options; kwargs...)

end # module
