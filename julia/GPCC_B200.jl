# GPCC_B200.jl -- drop-in Julia shim over libgpcc_b200.so (include/gpcc_b200.h).
#
# Keeps the public API of GPCC.jl v0.1.35 (src/GPCC.jl:30-31): `gpcc`, `getprobabilities`, `uniformpriordelay`, the
# returned `pred` closure (three methods) and `postb::MvNormal`, with identical signatures, and replaces the hot path
# (delayedCovariance.jl, gpccfixdelay_marginaliseb.jl:133-252, the README's map/pmap grid driver) by `ccall`s.
# NOTE: Julia is not available in the build environment of this repository, so this file has been written against the
# header but never executed; the same symbols are exercised through the Python ctypes mirror (gpcc_b200/api.py).
module GPCC_B200

using Distributions, LinearAlgebra, Random, Printf
import MiscUtil    # only to assert at load time that the library's transform formulas match MiscUtil's

export gpcc, gpccgrid, getprobabilities, uniformpriordelay, OU, rbf, matern32, matern52, statespace_fit_state

const LIB = get(ENV, "GPCC_B200_LIB", joinpath(@__DIR__, "..", "gpcc_b200", "libgpcc_b200.so"))

# the four kernels stay Julia functions (src/util.jl:15-52) so user code `kernel = GPCC.matern32` keeps working;
# the shim maps function identity to the C enum and errors on anything else (there is no CPU path).
OU(xi, xj; ρ = 1.0) = exp(-abs(xi - xj) / ρ)
rbf(xi, xj; ρ = 1.0) = exp(-0.5 * (xi - xj)^2 / (2ρ))
matern32(xi, xj; ρ = 1.0) = (r = abs(xi - xj); (1 + sqrt(3) * r / ρ) * exp(-sqrt(3) * r / ρ))
matern52(xi, xj; ρ = 1.0) = (r = abs(xi - xj); (1 + sqrt(5) * r / ρ + 5 * r^2 / (3 * ρ^2)) * exp(-sqrt(5) * r / ρ))
kernelid(k) = k === OU ? 0 : k === rbf ? 1 : k === matern32 ? 2 : k === matern52 ? 3 :
    error("GPCC_B200: unsupported kernel (expected OU, rbf, matern32 or matern52)")

struct FitOptions          # mirrors gpcc_fit_options (include/gpcc_b200.h), field for field
    max_iter::Cint; rhomin::Cdouble; rhomax::Cdouble; alpha_floor::Cdouble; gtol::Cdouble; ftol::Cdouble
    history::Cint; transform_id::Cint; theta0_per_candidate::Cint
    optimizer::Cint          # 0 = L-BFGS on the analytic gradient (default), 1 = Nelder-Mead on the device (the reference's, :205-211)
    nm_gtol::Cdouble         # Optim.Options(g_tol = 1e-6) (:205)
end

lasterror() = unsafe_string(ccall((:gpcc_last_error, LIB), Cstring, ()))
check(rc) = rc == 0 ? nothing : error("libgpcc_b200 error $rc: " * lasterror())

mutable struct Context
    h::Ptr{Cvoid}
    function Context(ndev::Integer = 1)
        r = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:gpcc_ctx_create, LIB), Cint, (Cint, Ptr{Cint}, Ref{Ptr{Cvoid}}), ndev, C_NULL, r))
        c = new(r[]); finalizer(c -> ccall((:gpcc_ctx_destroy, LIB), Cint, (Ptr{Cvoid},), c.h), c); c
    end
end
# One Julia process per GPU (`addprocs`, README.md:185-189): worker 1 draws the id with `communiqueid()`, the script sends the
# 128 bytes to the other workers (e.g. through `remotecall`), every worker calls `comminitrank!(ctx, nworkers, rank, id)`;
# from then on `gpccgrid` shards the grid over the workers' GPUs and all-gathers the results with NCCL.
function communiqueid()
    id = zeros(UInt8, 128)
    check(ccall((:gpcc_comm_unique_id, LIB), Cint, (Ptr{UInt8},), id)); id
end
comminitrank!(c::Context, world::Integer, rank::Integer, id::Vector{UInt8}) =
    check(ccall((:gpcc_ctx_comm_init_rank, LIB), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{UInt8}), c.h, world, rank, id))
const DEFAULT = Ref{Union{Nothing, Context}}(nothing)
defaultctx() = (DEFAULT[] === nothing && (DEFAULT[] = Context(parse(Int, get(ENV, "GPCC_B200_NDEV", "1")))); DEFAULT[])

mutable struct Problem
    h::Ptr{Cvoid}; L::Int; ctx::Context
    function Problem(ctx, tarray, yarray, stdarray, kernel)
        L = length(tarray); @assert L == length(yarray) == length(stdarray)          # gpccfixdelay_marginaliseb.jl:78
        n = Cint.(length.(tarray)); t = reduce(vcat, tarray); y = reduce(vcat, yarray); s = reduce(vcat, stdarray)
        μb = map(mean, yarray); Σb = 100 .* map(var, yarray)                          # :92-94, Julia's mean/var are authoritative
        r = Ref{Ptr{Cvoid}}(C_NULL)
        GC.@preserve n t y s μb Σb check(ccall((:gpcc_problem_create, LIB), Cint,
            (Ptr{Cvoid}, Cint, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Ptr{Cvoid}}),
            ctx.h, L, n, Float64.(t), Float64.(y), Float64.(s), kernelid(kernel), Float64.(μb), Float64.(Σb), r))
        p = new(r[], L, ctx); finalizer(p -> ccall((:gpcc_problem_destroy, LIB), Cint, (Ptr{Cvoid},), p.h), p); p
    end
end

# :dense factorises K + Sobs + B; :statespace (OU, matern32, matern52) runs the exact O(N) Kalman filter
# (gpcc_problem_set_method in include/gpcc_b200.h).  Fit states behind `pred` of `gpcc` are dense under either method;
# `statespace_fit_state` is the O(N) fit state of :statespace.
const METHODS = Dict(:dense => Cint(0), :statespace => Cint(1))
setmethod!(p::Problem, method::Symbol) =
    check(ccall((:gpcc_problem_set_method, LIB), Cint, (Ptr{Cvoid}, Cint), p.h, METHODS[method]))

function __init__()
    # the library hard-codes softplus / scaled logistic for MiscUtil.makepositive / transformbetween (transform_id 0)
    for x in (-3.0, 0.0, 2.5)
        @assert isapprox(MiscUtil.makepositive(x), log1p(exp(x)); rtol = 1e-12) "MiscUtil.makepositive is not softplus"
        @assert isapprox(MiscUtil.transformbetween(x, 0.1, 300.0), 0.1 + 299.9 / (1 + exp(-x)); rtol = 1e-12) "MiscUtil.transformbetween mismatch"
    end
end

# start points exactly as the reference draws them (gpccfixdelay_marginaliseb.jl:62, :160-176, :188-196)
function startpoints(yarray, seed, numberofrestarts, initialrandom, ρmin, ρmax)
    rg = MersenneTwister(seed); L = length(yarray)
    initialρ = numberofrestarts <= 2 ? rand(rg, Uniform(ρmin + 1e-3, ρmax - 1e-3), numberofrestarts) :
               collect(MiscUtil.logrange(ρmin + 1e-3, ρmax - 1e-3, numberofrestarts))
    θ0 = Array{Float64}(undef, L + 1, initialrandom, numberofrestarts)        # column-major == C [restart][draw][L+1]
    for i in 1:numberofrestarts, j in 1:initialrandom
        α = map(var, yarray) .* (rand(rg, L) * (1.2 - 0.8) .+ 0.8)
        θ0[:, j, i] = [MiscUtil.invmakepositive.(α); MiscUtil.invtransformbetween(initialρ[i], ρmin, ρmax)]
    end
    θ0, initialρ
end

options(iterations, ρmin, ρmax; percandidate = false, neldermead = false) =
    FitOptions(iterations, ρmin, ρmax, 1e-8, 1e-7, 1e-13, 8, 0, percandidate ? 1 : 0, neldermead ? 1 : 0, 1e-6)

# The state the reference's `pred` closures capture (:235-252): ONE factorisation per fitted (delays, alpha, rho), kept on the GPU.
mutable struct FitState
    h::Ptr{Cvoid}; p::Problem
    function FitState(p::Problem, d::Vector{Float64}, α::Vector{Float64}, ρ::Float64)
        r = Ref{Ptr{Cvoid}}(C_NULL)
        GC.@preserve d α check(ccall((:gpcc_fit_state_create, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Cdouble, Ref{Ptr{Cvoid}}), p.h, d, α, ρ, r))
        s = new(r[], p); finalizer(s -> ccall((:gpcc_fit_state_destroy, LIB), Cint, (Ptr{Cvoid},), s.h), s); s   # any destroy order is safe
    end
end

function fitbatch(p::Problem, delays::Matrix{Float64}, θ0, opt::FitOptions)     # delays: L x M (column per candidate)
    L, M = size(delays); P = size(θ0, 2)
    ll = zeros(M); θ = zeros(L + 1, M); α = zeros(L, M); ρ = zeros(M); it = zeros(Cint, M); nf = zeros(Cint, M); info = zeros(Cint, M)
    GC.@preserve delays θ0 ll θ α ρ it nf info check(ccall((:gpcc_fit_batch, LIB), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Ref{FitOptions}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cint}, Ptr{Cint}, Ptr{Cint}),
        p.h, M, delays, P, θ0, Ref(opt), ll, θ, α, ρ, it, nf, info))
    ll, α, ρ, info
end

"""
    loglikel, pred, (α, postb, ρ) = gpcc(tarray, yarray, stdarray; kernel, delays, iterations, seed = 1, numberofrestarts = 1, initialrandom = 5, rhomin = 0.1, rhomax, method = :dense)

Same contract as GPCC.gpcc (gpccfixdelay_marginaliseb.jl:46-53, 351).  `method = :statespace` (OU, matern32, matern52) fits with
the exact O(N) Kalman filter, takes postb from it, and factorises K + Sobs only when `pred` is first called.
"""
function gpcc(tarray, yarray, stdarray; kernel = kernel, delays = delays, iterations = iterations, seed = 1,
              numberofrestarts = 1, initialrandom = 5, rhomin = 0.1, rhomax = rhomax, neldermead = false, method = :dense)
    p = Problem(defaultctx(), tarray, yarray, stdarray, kernel); L = p.L
    method == :dense || setmethod!(p, method)
    @assert L == length(delays)
    Σb = 100 .* map(var, yarray)
    @printf("Running with random seed %d\n", seed)                                   # util.jl:1-11
    @printf("\t iterations             = %d\n\t initialrandom          = %d\n\t numberofrestarts       = %d\n", iterations, initialrandom, numberofrestarts)
    @printf("\t JITTER                 = %e\n\t ρmin                   = %f\n\t ρmax                   = %f\n", 1e-8, rhomin, rhomax)
    @printf("\t Σb                     = "); map(x -> @printf("%.3f ", x), Σb); @printf("\n")
    θ0, initialρ = startpoints(yarray, seed, numberofrestarts, initialrandom, rhomin, rhomax)
    @printf("\n\tInitial ρ values are:\n"); map(x -> @printf("\t%f\n", x), initialρ)
    τ = repeat(Float64.(delays), 1, numberofrestarts)                                # one "candidate" per restart (:222-226)
    ll, αs, ρs, _ = fitbatch(p, τ, θ0, options(iterations, rhomin, rhomax; percandidate = true, neldermead = neldermead))
    b = argmax(ll); α = αs[:, b]; ρ = ρs[b]
    @printf("\n\tOverall minimum is %f\n", -ll[b]); @show α, ρ                        # :228, :235
    d = Float64.(delays); μ = zeros(L); Σ = zeros(L, L)
    stref = Ref{Union{Nothing, FitState}}(nothing)
    state() = (stref[] === nothing && (stref[] = FitState(p, d, α, ρ)); stref[])   # K, KSobsB (:237-241): factorised once
    if method == :statespace          # postb from the filter; the factorisation waits for the first prediction
        GC.@preserve d α μ Σ check(ccall((:gpcc_postb, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Cdouble, Ptr{Cdouble}, Ptr{Cdouble}), p.h, d, α, ρ, μ, Σ))
    else
        GC.@preserve μ Σ check(ccall((:gpcc_fit_state_postb, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}), state().h, μ, Σ))
    end
    postb = MvNormal(μ, Symmetric(Σ))                                                # :252

    function predictTest(ttest::Union{Array{Array{Float64, 1}, 1}, Array{T} where T <: AbstractRange{S} where S <: Real})   # :259-289
        nt = Cint.(length.(ttest)); tt = Float64.(reduce(vcat, collect.(ttest))); NT = length(tt)
        μp = zeros(NT); Σp = zeros(NT, NT)
        GC.@preserve nt tt μp Σp check(ccall((:gpcc_fit_state_predict, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), state().h, nt, tt, μp, C_NULL, Σp))
        μp, Σp
    end
    function predictTest(ttest::Union{AbstractRange{Float64}, Array{Float64, 1}})                                          # :293-307
        Nt = length(ttest); nt = fill(Cint(Nt), L); tt = repeat(Float64.(collect(ttest)), L); μp = zeros(L * Nt); σp = zeros(L * Nt)
        GC.@preserve nt tt μp σp check(ccall((:gpcc_fit_state_predict, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), state().h, nt, tt, μp, σp, C_NULL))
        [μp[idx] for idx in Iterators.partition(1:L*Nt, Nt)], [σp[idx] for idx in Iterators.partition(1:L*Nt, Nt)]
    end
    function predictTest(ttest::Array{Array{Float64, 1}, 1}, ytest::Array{Array{Float64, 1}, 1}, σtest::Array{Array{Float64, 1}, 1})   # :311-343
        nt = Cint.(length.(ttest)); tt = reduce(vcat, ttest); yt = reduce(vcat, ytest); σt = reduce(vcat, σtest)
        ll_ = Ref{Cdouble}(0.0); info = Ref{Cint}(0)
        GC.@preserve nt tt yt σt check(ccall((:gpcc_fit_state_predict_loglik, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cdouble}, Ref{Cint}), state().h, nt, tt, yt, σt, ll_, info))
        if info[] != 0      # PosDefException branch (:327-333): repair on the host exactly as the reference does
            μp, Σp = predictTest(ttest); Σp = Σp + Diagonal(σt .^ 2)
            return logpdf(MvNormal(μp, MiscUtil.nearestposdef(MiscUtil.makematrixsymmetric(Σp); minimumeigenvalue = 1e-6)), yt)
        end
        ll_[]
    end
    ll[b], predictTest, (α, postb, ρ)
end

# The O(N) fit state of the state-space method (gpcc_ss_state_*): filtered moments and backward-pass adjoint, no N x N matrix.
mutable struct SSFitState
    h::Ptr{Cvoid}; p::Problem
    function SSFitState(p::Problem, d::Vector{Float64}, α::Vector{Float64}, ρ::Float64)
        r = Ref{Ptr{Cvoid}}(C_NULL)
        GC.@preserve d α check(ccall((:gpcc_ss_state_create, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Cdouble, Ref{Ptr{Cvoid}}), p.h, d, α, ρ, r))
        s = new(r[], p); finalizer(s -> ccall((:gpcc_ss_state_destroy, LIB), Cint, (Ptr{Cvoid},), s.h), s); s   # the state owns its data
    end
end

"""
    pred = statespace_fit_state(tarray, yarray, stdarray; kernel, delays, α, ρ)

`pred` at fixed (delays, α, ρ) from the O(N) fit state of the state-space method (OU, matern32, matern52): `pred(ttest)`
gives per band (μ, σ) (:293-307) and `pred(ttest, ytest, σtest)` the test log-likelihood (:311-343), for light curves far
beyond a dense factorisation.  The full predictive covariance (`pred(::Vector{Vector})`) needs the dense state of `gpcc`.
"""
function statespace_fit_state(tarray, yarray, stdarray; kernel = kernel, delays = delays, α = α, ρ = ρ)
    p = Problem(defaultctx(), tarray, yarray, stdarray, kernel); L = p.L
    setmethod!(p, :statespace)
    st = SSFitState(p, Float64.(delays), Float64.(α), Float64(ρ))
    function predictTest(ttest::Union{AbstractRange{Float64}, Array{Float64, 1}})                                          # :293-307
        Nt = length(ttest); nt = fill(Cint(Nt), L); tt = repeat(Float64.(collect(ttest)), L); μp = zeros(L * Nt); σp = zeros(L * Nt)
        GC.@preserve nt tt μp σp check(ccall((:gpcc_ss_state_predict, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), st.h, nt, tt, μp, σp))
        [μp[idx] for idx in Iterators.partition(1:L*Nt, Nt)], [σp[idx] for idx in Iterators.partition(1:L*Nt, Nt)]
    end
    predictTest(ttest::Array{Array{Float64, 1}, 1}) =
        error("the state-space fit state gives per-point means and standard deviations: the full predictive covariance needs the dense state of gpcc")
    function predictTest(ttest::Array{Array{Float64, 1}, 1}, ytest::Array{Array{Float64, 1}, 1}, σtest::Array{Array{Float64, 1}, 1})   # :311-343
        nt = Cint.(length.(ttest)); tt = reduce(vcat, ttest); yt = reduce(vcat, ytest); σt = reduce(vcat, σtest)
        ll_ = Ref{Cdouble}(0.0); info = Ref{Cint}(0)
        GC.@preserve nt tt yt σt check(ccall((:gpcc_ss_state_predict_loglik, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cdouble}, Ref{Cint}), st.h, nt, tt, yt, σt, ll_, info))
        info[] == 0 || error("non-positive innovation variance at merged position $(info[]): the nearestposdef repair needs the dense state of gpcc")
        ll_[]
    end
    predictTest
end

"""
    gpccgrid(tarray, yarray, stdarray, candidatedelays; kernel, iterations, rhomax, ...) -> (loglikel, posterior, α, ρ)

Batched replacement of the README's `map`/`pmap` idiom (README.md:170-210, 285): `candidatedelays` is a vector of
L-vectors; the grid is sharded over the context's GPUs, log-likelihoods are all-gathered with NCCL and normalised.
"""
function gpccgrid(tarray, yarray, stdarray, candidatedelays; kernel = kernel, iterations = iterations, seed = 1, initialrandom = 5,
                  rhomin = 0.1, rhomax = rhomax, logprior = nothing, method = :dense)
    p = Problem(defaultctx(), tarray, yarray, stdarray, kernel); L = p.L; M = length(candidatedelays)
    method == :dense || setmethod!(p, method)
    τ = Float64.(reduce(hcat, candidatedelays)); θ0, _ = startpoints(yarray, seed, 1, initialrandom, rhomin, rhomax)
    ll = zeros(M); post = zeros(M); α = zeros(L, M); ρ = zeros(M); lp = logprior === nothing ? C_NULL : Float64.(vec(logprior))
    GC.@preserve τ θ0 ll post α ρ lp check(ccall((:gpcc_grid_posterior, LIB), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Ref{FitOptions}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cint}, Ptr{Cint}),
        p.h, M, τ, lp, initialrandom, θ0[:, :, 1], Ref(options(iterations, rhomin, rhomax)), ll, post, C_NULL, α, ρ, C_NULL, C_NULL))
    ll, post, α, ρ
end

# src/getprobabilities.jl:1-20 -- shape preserving
getprobabilities(loglikel) = getprobabilities(loglikel, ones(size(loglikel)))
function getprobabilities(loglikel, logpriorpdfvalues)
    ll = Float64.(vec(loglikel)); lp = Float64.(vec(logpriorpdfvalues)); out = similar(ll)
    GC.@preserve ll lp out check(ccall((:gpcc_getprobabilities, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), defaultctx().h, length(ll), ll, lp, out))
    reshape(out, size(loglikel))
end

# src/uniformpriordelay.jl:10-16 -- scalar host arithmetic, unchanged
uniformpriordelay(; L = L, z = z) = Uniform(0.0, 10.0^(1.559) * (L * 10^(-44))^(0.549) * (1 + z))

end # module
