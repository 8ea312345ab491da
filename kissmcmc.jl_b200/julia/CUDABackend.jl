# KissMCMC.CUDABackend -- thin `ccall` layer over libkissmcmc_cuda.so (include/kissmcmc_cuda.h).
#
# Drop this file next to src/samplers.jl of KissMCMC.jl and add `include("CUDABackend.jl")` to
# src/KissMCMC.jl (after line 11).  It keeps the reference's call shapes
#
#     emcee(logdensity, theta0s; niter, nburnin, nthin, a_scale, use_progress_meter, hasblob, ...)
#     make_theta0s(theta0, ball_radius, logdensity, nwalkers; ...)
#     squash_walkers(thetas, accept_ratio, logdensities, blobs; ...)   (unchanged: host side)
#     metropolis(logdensity, sample_ppdf, theta0; niter, nburnin, nthin, ...)
#
# with ONE difference: `logdensity` is a `LogDensity` plugin descriptor instead of a closure (and metropolis's
# `sample_ppdf` a `NormalProposal` or `MvNormalProposal`)
# (closures cannot cross the C-ABI onto the GPU; there is no CPU fallback and no CUDA.jl).
#
# NOTE: Julia is not installed in the build image, so this module has not been executed
# there; the identical C-ABI is exercised by the Python ctypes harness (kissmcmc.jl_b200/api.py)
# and the GPU parity tests.
module CUDABackend

export LogDensity, exponential, rosenbrock, gaussian, gaussian_mixture, lognormal, logistic, set_option!, info, emcee, emcee_squashed,
       make_theta0s, g_pdf, cdf_g_inv, sample_g, NormalProposal, MvNormalProposal, normal_proposal, metropolis

using LinearAlgebra: cholesky, Symmetric, diag, inv
import ..KissMCMC: squash_walkers   # host-side, reused as is (src/samplers.jl:372-428)

# The library name of every `ccall((:sym, LIB[]), ...)` is an expression evaluated at the first call: this needs
# Julia >= 1.6 (the reference's Project.toml allows 1.2; on older versions make LIB a `const String`).
const LIB = Ref{String}(get(ENV, "KISSMCMC_CUDA_LIB", "libkissmcmc_cuda"))

const MODE_PHILOX = Int32(0)
const MODE_REPLAY = Int32(1)
const MULTI_SHARDED = Int32(0)       # ONE ensemble sharded by walker index over the devices
const MULTI_INDEPENDENT = Int32(1)   # one independent ensemble per device

struct KmcError <: Exception
    code::Int32
    msg::String
end
Base.showerror(io::IO, e::KmcError) = print(io, "libkissmcmc_cuda error $(e.code): $(e.msg)")

last_error() = unsafe_string(ccall((:kmc_last_error, LIB[]), Cstring, ()))
check(rc::Int32) = rc == 0 ? nothing : throw(KmcError(rc, last_error()))

# mirrors `struct kmc_emcee_opts` field for field
struct EmceeOpts
    niter_walker::Int64
    nburnin_walker::Int64
    nthin::Int64
    a_scale::Float64
    seed::UInt64
    mode::Int32
    device::Int32
    walker_id_base::Int64
    launch_mode::Int32
    exchange::Int32
    shard_begin::Int64
    shard_count::Int64
    push_chunk::Int32
    push_cap::Int32
    push_lag::Int32
    reserved::Int32
end

# ------------------------------------------------------------------ log-density plugins
"A device log-density plugin instance (replaces the closure `pdf`, src/samplers.jl:257)."
mutable struct LogDensity
    handle::Ptr{Cvoid}
    name::String
    d::Int
    device::Int          # the device that holds the plugin's parameters / data: emcee runs there by default
    function LogDensity(name::AbstractString, d::Integer, params::Vector{Float64}=Float64[];
                        data::Union{Nothing,Array}=nothing, device::Integer=0)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        dptr = data === nothing ? C_NULL : pointer(data)
        dbytes = data === nothing ? 0 : sizeof(data)
        GC.@preserve params data check(ccall((:kmc_density_create, LIB[]), Int32,
            (Cstring, Int32, Ptr{Float64}, Int64, Ptr{Cvoid}, Int64, Int32, Ref{Ptr{Cvoid}}),
            name, d, params, length(params), dptr, dbytes, device, h))
        obj = new(h[], String(name), Int(d), Int(device))
        finalizer(o -> ccall((:kmc_density_destroy, LIB[]), Int32, (Ptr{Cvoid},), o.handle), obj)
        return obj
    end
end

"README.md:15  `logpdf(x) = x<0 ? -Inf : -x`"
exponential(d::Integer=1; device=0) = LogDensity("exponential", d; device=device)
"test/runtests.jl:68  `-(b*(x[2]-x[1]^2)^2 + (a-x[1])^2)/temper`"
rosenbrock(a=1.0, b=100.0, temper=20.0; device=0) = LogDensity("rosenbrock", 2, Float64[a, b, temper]; device=device)
"MvNormal(mean, cov) (test/runtests.jl:53,61): params = [mu; vec(A'); lognorm], A = chol(inv(cov))' so that |A(x-mu)|^2 is the Mahalanobis form"
function gaussian(mean, cov; device=0)
    mu = Float64.(vcat(mean))
    d = length(mu)
    prec = inv(reshape(Float64.(collect(cov)), d, d))
    Lc = cholesky(Symmetric((prec + prec') / 2)).L          # prec = L L'
    A = Matrix(Lc')                                          # y = A (x - mu)
    lognorm = sum(log.(diag(Lc))) - 0.5 * d * log(2pi)
    params = vcat(mu, vec(permutedims(A)), lognorm)          # A row-major
    return LogDensity("gaussian", d, params; device=device)
end
"""
    gaussian_mixture(weights, means, covs; device=0)

`MixtureModel(MvNormal.(means, covs), weights)`: `weights` (K, each > 0, normalised here), `means` (K vectors of length
d, or K numbers for d = 1), `covs` (K symmetric positive definite d x d matrices, or K variances for d = 1).
params = per component [mu_k; upper triangle of A_k = chol(inv(Sigma_k))' row by row; log(w_k / sum w) + lognorm_k],
the per-component math of `gaussian`.  Fused kernels for d in {1..6, 8, 10, 12, 16} with K <= Kmax(d) =
floor(272 / (d + d(d+1)/2 + 1)): 90, 45, 27, 18, 12, 9, 6, 4, 2, 1 (KmcError 3 otherwise).  Like the rest of this
module it has not been executed (no Julia in the build image); the Python `gaussian_mixture` packs the same layout.
"""
function gaussian_mixture(weights, means, covs; device=0)
    K = length(weights)
    (length(means) == K && length(covs) == K) || throw(ArgumentError("weights, means and covs need one entry per component"))
    all(w -> isfinite(w) && w > 0, weights) || throw(ArgumentError("every weight must be finite and > 0"))
    total = sum(Float64.(weights))
    d = length(vcat(means[1]))
    params = Float64[]
    for k in 1:K
        mu = Float64.(vcat(means[k]))
        length(mu) == d || throw(ArgumentError("component $(k - 1): mean has length $(length(mu)), expected $d"))
        prec = inv(reshape(Float64.(collect(covs[k])), d, d))
        Lc = cholesky(Symmetric((prec + prec') / 2)).L      # prec = L L'
        A = Matrix(Lc')                                      # upper triangular, y = A (x - mu)
        lognorm = sum(log.(diag(Lc))) - 0.5 * d * log(2pi)
        append!(params, mu)
        for i in 1:d, j in i:d                               # row by row, j = i .. d
            push!(params, A[i, j])
        end
        push!(params, log(weights[k] / total) + lognorm)
    end
    return LogDensity("gaussian_mixture", d, params; device=device)
end
"LogNormal(mu, sigma) (test/runtests.jl:56)"
lognormal(mu=0.0, sigma=1.0; device=0) =
    LogDensity("lognormal", 1, Float64[mu, sigma, log(sigma) + 0.5 * log(2pi)]; device=device)

"""
    logistic(X, y; prior_sigma=10.0, device=0, tensor_cores=false)

Bayesian logistic regression (BASELINE.json configs[3]): `X` is N x d, `y` in {0,1}, prior N(0, sigma^2 I).
Exact FP64 by default; `tensor_cores=true` opts in to the tcgen05 kernel (d <= 64 and bf16-representable X; FP64: any d <= 512), which is
approximate, with an error that grows with the size of the logits: per point, with u = 2^-24 and m = ceil(d/16),
`|logp - logp_fp64| <= u [(0.5 + 1.05 m) sum_n sum_k |theta_k x_nk| + 8.5 sum_n |theta . x_n|] + 5 u N`, and the sum of
two points' bounds on their difference.  At d = 32, N = 10^6, theta* ~ N(0, 1/d) that is ~1.3 per point (a B200 shows
a common offset of ~3e-8 N and 2e-3 on differences); with the data drawn from 16 theta*, ~13.
"""
function logistic(X::AbstractMatrix, y::AbstractVector; prior_sigma=10.0, device=0, tensor_cores=false)
    N, d = size(X)
    @assert length(y) == N
    data = vcat(vec(permutedims(Float32.(X))), Float32.(y))          # float32 X[N][d] row-major, then y[N]
    ld = LogDensity("logistic", d, Float64[prior_sigma]; data=data, device=device)
    tensor_cores && set_option!(ld, "tensor_cores", 1)
    return ld
end

"Plugin options (`\"tensor_cores\"`, `\"fused_variant\"`): see include/kissmcmc_cuda.h."
set_option!(ld::LogDensity, key::AbstractString, value::Real) =
    check(ccall((:kmc_density_set_option, LIB[]), Int32, (Ptr{Cvoid}, Cstring, Float64), ld.handle, key, value))
function info(ld::LogDensity, key::AbstractString)
    v = Ref{Float64}(0)
    check(ccall((:kmc_density_get_info, LIB[]), Int32, (Ptr{Cvoid}, Cstring, Ref{Float64}), ld.handle, key, v))
    return v[]
end

# ------------------------------------------------------------------ g distribution (src/samplers.jl:223-230)
"src/samplers.jl:224"
function g_pdf(z::Real, a::Real)
    zz, out = Float64[z], Float64[0]
    check(ccall((:kmc_g_pdf, LIB[]), Int32, (Ptr{Float64}, Int64, Float64, Ptr{Float64}), zz, 1, a, out))
    return out[1]
end
"src/samplers.jl:227"
function cdf_g_inv(u::Real, a::Real)
    uu, out = Float64[u], Float64[0]
    check(ccall((:kmc_cdf_g_inv, LIB[]), Int32, (Ptr{Float64}, Int64, Float64, Ptr{Float64}), uu, 1, a, out))
    return out[1]
end
"src/samplers.jl:230: `n` draws of z ~ g on the device, through the sampler's own draw path"
function sample_g(a::Real, n::Integer=1; seed::Integer=0, device::Integer=0)
    out = Vector{Float64}(undef, n)
    check(ccall((:kmc_sample_g, LIB[]), Int32, (Float64, UInt64, Int64, Int32, Ptr{Float64}), a, seed, n, device, out))
    return n == 1 ? out[1] : out
end

"Batched evaluation: `thetas` is d x n (column = one point); returns n log-densities."
function (ld::LogDensity)(thetas::AbstractMatrix{Float64})
    @assert size(thetas, 1) == ld.d
    th = Matrix{Float64}(thetas)
    out = Vector{Float64}(undef, size(th, 2))
    GC.@preserve th out check(ccall((:kmc_density_eval, LIB[]), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}), ld.handle, th, size(th, 2), out))
    return out
end
(ld::LogDensity)(theta::AbstractVector{<:Real}) = ld(reshape(Float64.(theta), ld.d, 1))[1]
(ld::LogDensity)(theta::Real) = ld(reshape(Float64[theta], 1, 1))[1]

# ------------------------------------------------------------------ emcee (src/samplers.jl:188-216)
to_matrix(theta0s::AbstractVector{<:Real}) = reshape(Float64.(theta0s), 1, :)
to_matrix(theta0s::AbstractVector) = Float64.(reduce(hcat, theta0s))      # d x nw, column-major

"""
    emcee(logdensity::LogDensity, theta0s; niter=10^5, nburnin=niter÷2, nthin=1, a_scale=2.0,
          use_progress_meter=true, hasblob=false, seed=0, replay=nothing)

Same semantics and 4-tuple as `KissMCMC.emcee`: `(thetas, accept_ratio, logdensities, nothing)`
with `thetas::Vector{Vector{T}}` (one chain per walker).  `replay=(partner, z, u)` uploads the
draws (partner = 1-based walker index as in Julia; converted to 0-based for the ABI).
"""
function emcee(ld::LogDensity, theta0s; niter=10^5, nburnin=niter ÷ 2, nthin=1, a_scale=2.0,
               use_progress_meter=true, hasblob=false, init_blobs=nothing, reduce_blob! =nothing,
               seed::Integer=0, replay=nothing, device::Integer=ld.device, devices=nothing, sharded::Bool=true)
    hasblob && error("hasblob=true is not supported by the CUDA backend (blobs are host objects)")
    if devices !== nothing                                                  # several GPUs of this process
        replay === nothing || error("replay mode runs on one device")
        return emcee_multi(ld, theta0s, collect(Int32, devices), sharded; niter=niter, nburnin=nburnin, nthin=nthin,
                           a_scale=a_scale, seed=seed)
    end
    x0 = to_matrix(deepcopy(theta0s))                                       # :198
    @assert a_scale > 1                                                     # :200
    nwalkers = size(x0, 2)
    @assert iseven(nwalkers) "Use an even number of walkers."               # :202
    niter_walker = niter ÷ nwalkers                                         # :203
    nburnin_walker = nburnin ÷ nwalkers                                     # :204
    d = size(x0, 1)
    @assert nwalkers >= d + 2 "Use more walkers: at least DOF+2, but better many more."   # :205

    opts = Ref(EmceeOpts(niter_walker, nburnin_walker, nthin, a_scale, UInt64(seed),
                         replay === nothing ? MODE_PHILOX : MODE_REPLAY, device, 0, 0, 0, 0, 0, 0, 0, 0, 0))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve x0 check(ccall((:kmc_emcee_create, LIB[]), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ref{EmceeOpts}, Ref{Ptr{Cvoid}}),
        ld.handle, x0, nwalkers, d, opts, h))
    s = h[]
    try
        if replay !== nothing
            partner = Int64.(replay[1]) .- 1
            z, u = Float64.(replay[2]), Float64.(replay[3])
            GC.@preserve partner z u check(ccall((:kmc_emcee_set_replay, LIB[]), Int32,
                (Ptr{Cvoid}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Int64),
                s, partner, z, u, length(partner) ÷ nwalkers))
        end
        if use_progress_meter && niter_walker > 0          # coarse: at most 20 polls, never per iteration
            done = 0
            for c in 1:min(20, niter_walker)
                upto = (niter_walker * c) ÷ min(20, niter_walker)
                check(ccall((:kmc_emcee_run, LIB[]), Int32, (Ptr{Cvoid}, Int64), s, upto - done))
                done = upto
                it, m, sd, outl = Ref{Int64}(0), Ref{Float64}(0), Ref{Float64}(0), Ref{Int64}(0)
                check(ccall((:kmc_emcee_progress, LIB[]), Int32,
                    (Ptr{Cvoid}, Ref{Int64}, Ref{Float64}, Ref{Float64}, Ref{Int64}), s, it, m, sd, outl))
                nn = max(1, it[] > nburnin_walker ? it[] - nburnin_walker : it[])
                print(stderr, "\remcee, niter=$niter, nwalkers=$nwalkers: $(100done ÷ niter_walker)%  ",
                      "accept_ratio_mean=$(round(m[]/nn, sigdigits=3)) accept_ratio_std=$(round(sd[]/nn, sigdigits=3)) ",
                      "accept_ratio_outliers=$(outl[]) burnin_phase=$(it[] <= nburnin_walker)")
            end
            println(stderr)
        else
            check(ccall((:kmc_emcee_run, LIB[]), Int32, (Ptr{Cvoid}, Int64), s, -1))
        end
        nsr = Ref{Int64}(0)
        check(ccall((:kmc_emcee_nsamples, LIB[]), Int32, (Ptr{Cvoid}, Ref{Int64}), s, nsr))
        ns = nsr[]
        th = Array{Float64,3}(undef, d, ns, nwalkers)       # (ntheta, nsamples, nchains), src/analysis.jl:143
        lp = Matrix{Float64}(undef, ns, nwalkers)
        ar = Vector{Float64}(undef, nwalkers)
        GC.@preserve th lp ar check(ccall((:kmc_emcee_copy_results, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), s, th, lp, ar))
        scalar = eltype(theta0s) <: Real
        thetas = scalar ? [th[1, :, w] for w in 1:nwalkers] :
                          [[th[:, i, w] for i in 1:ns] for w in 1:nwalkers]
        logdensities = [lp[:, w] for w in 1:nwalkers]
        return thetas, ar, logdensities, nothing            # blobs: nothing (:221, test/emcee.jl:33)
    finally
        ccall((:kmc_emcee_destroy, LIB[]), Int32, (Ptr{Cvoid},), s)
    end
end

"""
    emcee_multi(ld, theta0s, devices, sharded; niter, nburnin, nthin, a_scale, seed)

Library-owned multi-GPU (`emcee(...; devices=0:7, sharded=true)`): `sharded=true` shards ONE ensemble by walker index
over `devices` -- the owners of the passive half push the packed partner rows each peer's walkers will ask for over
NVLink, no collective, no cross-GPU barrier -- and returns exactly the chains of the single-GPU run; `sharded=false` runs
one independent ensemble per device from `theta0s[r]` (a vector of ensembles) and concatenates them.
Replaces, across GPUs, the threaded sweep of src/samplers.jl:246-273.
"""
function emcee_multi(ld::LogDensity, theta0s, devices::Vector{Int32}, sharded::Bool; niter=10^5, nburnin=niter ÷ 2,
                     nthin=1, a_scale=2.0, seed::Integer=0)
    ndev = length(devices)
    x0 = sharded ? to_matrix(deepcopy(theta0s)) : reduce(hcat, [to_matrix(deepcopy(t)) for t in theta0s])
    d = size(x0, 1)
    nwalkers = sharded ? size(x0, 2) : size(x0, 2) ÷ ndev
    @assert a_scale > 1
    @assert iseven(nwalkers) "Use an even number of walkers."
    @assert nwalkers >= d + 2 "Use more walkers: at least DOF+2, but better many more."
    opts = Ref(EmceeOpts(niter ÷ nwalkers, nburnin ÷ nwalkers, nthin, a_scale, UInt64(seed), MODE_PHILOX, 0, 0, 0, 0, 0,
                         0, 0, 0, 0, 0))
    handles = fill(ld.handle, ndev)                       # fused plugins keep no device memory: one handle serves all
    m = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve x0 handles devices check(ccall((:kmc_emcee_create_multi, LIB[]), Int32,
        (Ptr{Ptr{Cvoid}}, Ptr{Float64}, Int64, Int32, Ref{EmceeOpts}, Ptr{Int32}, Int32, Int32, Ref{Ptr{Cvoid}}),
        handles, x0, nwalkers, d, opts, devices, ndev, sharded ? MULTI_SHARDED : MULTI_INDEPENDENT, m))
    try
        check(ccall((:kmc_multi_run, LIB[]), Int32, (Ptr{Cvoid}, Int64), m[], -1))
        check(ccall((:kmc_multi_sync, LIB[]), Int32, (Ptr{Cvoid},), m[]))
        nsr, nwr = Ref{Int64}(0), Ref{Int64}(0)
        check(ccall((:kmc_multi_shape, LIB[]), Int32, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}), m[], nsr, nwr))
        ns, nwo = nsr[], nwr[]
        th = Array{Float64,3}(undef, d, ns, nwo)
        lp = Matrix{Float64}(undef, ns, nwo)
        ar = Vector{Float64}(undef, nwo)
        GC.@preserve th lp ar check(ccall((:kmc_multi_copy_results, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), m[], th, lp, ar))
        first = sharded ? theta0s : theta0s[1]
        scalar = eltype(first) <: Real
        thetas = scalar ? [th[1, :, w] for w in 1:nwo] : [[th[:, i, w] for i in 1:ns] for w in 1:nwo]
        return thetas, ar, [lp[:, w] for w in 1:nwo], nothing
    finally
        ccall((:kmc_multi_destroy, LIB[]), Int32, (Ptr{Cvoid},), m[])
    end
end

"""
    emcee_squashed(ld, theta0s; niter, nburnin, nthin, a_scale, seed, drop_low_accept_ratio=false, drop_fact=2, order=false)

`squash_walkers(emcee(...)...)` (src/samplers.jl:372-428) with the squash done ON THE DEVICE: the per-walker chains
never cross PCIe un-squashed.  Returns `(thetas, mean_accept_ratio, logdensities, nothing)` like `squash_walkers`.
"""
function emcee_squashed(ld::LogDensity, theta0s; niter=10^5, nburnin=niter ÷ 2, nthin=1, a_scale=2.0, seed::Integer=0,
                        drop_low_accept_ratio=false, drop_fact=2, order=false, device::Integer=ld.device)
    x0 = to_matrix(deepcopy(theta0s))
    d, nwalkers = size(x0)
    @assert a_scale > 1
    @assert iseven(nwalkers) "Use an even number of walkers."
    @assert nwalkers >= d + 2 "Use more walkers: at least DOF+2, but better many more."
    opts = Ref(EmceeOpts(niter ÷ nwalkers, nburnin ÷ nwalkers, nthin, a_scale, UInt64(seed), MODE_PHILOX, device, 0, 0, 0,
                         0, 0, 0, 0, 0, 0))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve x0 check(ccall((:kmc_emcee_create, LIB[]), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ref{EmceeOpts}, Ref{Ptr{Cvoid}}), ld.handle, x0, nwalkers, d, opts, h))
    s = h[]
    try
        check(ccall((:kmc_emcee_run, LIB[]), Int32, (Ptr{Cvoid}, Int64), s, -1))
        nsr = Ref{Int64}(0)
        check(ccall((:kmc_emcee_nsamples, LIB[]), Int32, (Ptr{Cvoid}, Ref{Int64}), s, nsr))
        nk, am, med, sd = Ref{Int64}(0), Ref{Float64}(0), Ref{Float64}(0), Ref{Float64}(0)
        sq(th, lp) = check(ccall((:kmc_emcee_squash, LIB[]), Int32,
            (Ptr{Cvoid}, Int32, Float64, Int32, Ptr{Float64}, Ptr{Float64}, Ref{Int64}, Ref{Float64}, Ref{Float64}, Ref{Float64}),
            s, drop_low_accept_ratio ? 1 : 0, drop_fact, order ? 1 : 0, th, lp, nk, am, med, sd))
        sq(C_NULL, C_NULL)                                   # sizes first
        th = Matrix{Float64}(undef, d, nk[] * nsr[])
        lp = Vector{Float64}(undef, nk[] * nsr[])
        GC.@preserve th lp sq(pointer(th), pointer(lp))
        scalar = eltype(theta0s) <: Real
        thetas = scalar ? vec(th) : [th[:, i] for i in 1:size(th, 2)]
        return thetas, am[], lp, nothing
    finally
        ccall((:kmc_emcee_destroy, LIB[]), Int32, (Ptr{Cvoid},), s)
    end
end

# ------------------------------------------------------------------ make_theta0s (src/samplers.jl:311-349)
"""
    make_theta0s(theta0, ball_radius, logdensity::LogDensity, nwalkers; ball_radius_halfing_steps=7, ntries=100, seed=0)

Reference loop semantics (including the cumulative radius halving of :326 and the silent skip of a walker that
exhausts every try) ON THE DEVICE: counter-based Philox / Box-Muller normals, rejection of points whose plugin
log-density is not > -Inf (:338), all pending walkers tried at once.
"""
function make_theta0s(theta0::T, ball_radius, ld::LogDensity, nwalkers; ball_radius_halfing_steps=7, ntries=100,
                      hasblob=false, seed::Integer=0) where T
    hasblob && error("hasblob=true is not supported by the CUDA backend")
    npara = length(theta0)
    br = ball_radius isa Number ? ones(npara) * ball_radius : Float64.(collect(ball_radius))   # :316-318
    @assert length(br) == npara                                                                # :319
    th0 = Float64.(vcat(theta0))
    out = Matrix{Float64}(undef, npara, nwalkers)
    nf = Ref{Int64}(0)
    GC.@preserve th0 br out check(ccall((:kmc_make_theta0s, LIB[]), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Int32, Int32, UInt64, Ptr{Float64}, Ref{Int64}),
        ld.handle, th0, br, nwalkers, ball_radius_halfing_steps, ntries, seed, out, nf))
    return T <: Number ? [out[1, c] for c in 1:nf[]] : [T(out[:, c]) for c in 1:nf[]]
end

# ------------------------------------------------------------------ metropolis (src/samplers.jl:9-128)
"Symmetric Gaussian random walk `theta1 = theta0 .+ sigma .* randn(d)` in place of the closure `sample_ppdf`."
struct NormalProposal
    sigma::Vector{Float64}       # one scale, or one per component; finite and > 0 (checked by the library)
end
normal_proposal(sigma::Real) = NormalProposal(Float64[sigma])
normal_proposal(sigma::AbstractVector{<:Real}) = NormalProposal(Float64.(sigma))

"Correlated Gaussian random walk `theta1 = theta0 .+ L * randn(d)`, L the lower Cholesky factor of the covariance."
struct MvNormalProposal
    chol::Matrix{Float64}        # the column-major UPPER factor U = L': its memory is L row-major, as the library takes it
end
normal_proposal(Sigma::AbstractMatrix{<:Real}) = MvNormalProposal(Matrix{Float64}(cholesky(Symmetric(Float64.(Sigma))).U))

# kmc_metropolis_create(_chol) for either proposal
create_metropolis(ld, x0, k, d, p::NormalProposal, opts, h) =
    GC.@preserve x0 p check(ccall((:kmc_metropolis_create, LIB[]), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ptr{Float64}, Int64, Ref{EmceeOpts}, Ref{Ptr{Cvoid}}),
        ld.handle, x0, k, d, p.sigma, length(p.sigma), opts, h))
function create_metropolis(ld, x0, k, d, p::MvNormalProposal, opts, h)
    size(p.chol) == (d, d) || error("the proposal's Cholesky factor is $(size(p.chol)), the density has d=$d")
    GC.@preserve x0 p check(ccall((:kmc_metropolis_create_chol, LIB[]), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ptr{Float64}, Ref{EmceeOpts}, Ref{Ptr{Cvoid}}),
        ld.handle, x0, k, d, p.chol, opts, h))
end

"""
    metropolis(logdensity::LogDensity, proposal, theta0; niter=10^5, nburnin=niter÷2, nthin=1,
               use_progress_meter=true, hasblob=false, seed=0, nchains=nothing, device=logdensity.device)

`proposal` is `normal_proposal(sigma)` (diagonal) or `normal_proposal(Sigma::AbstractMatrix)` (correlated, factored
with `cholesky`).

Same semantics and 4-tuple as `KissMCMC.metropolis`: `(thetas::Vector{T}, accept_ratio::Float64,
logdensities::Vector{Float64}, nothing)`; `niter` counts the steps of one chain.  With `nchains=k`, `theta0` is a
vector of k starting points and every element of the tuple holds one entry per independent chain (chain c draws
with id c - 1, so it is the same chain whatever k is).
"""
function metropolis(ld::LogDensity, proposal::Union{NormalProposal,MvNormalProposal}, theta0; niter=10^5,
                    nburnin=niter ÷ 2, nthin=1, use_progress_meter=true, hasblob=false, seed::Integer=0,
                    nchains=nothing, device::Integer=ld.device)
    hasblob && error("hasblob=true is not supported by the CUDA backend (blobs are host objects)")
    starts = nchains === nothing ? [deepcopy(theta0)] : deepcopy(theta0)
    nchains === nothing || @assert length(starts) == nchains "theta0 must hold nchains starting points"
    x0 = to_matrix(starts)                                                  # d x nchains
    d, k = size(x0)
    opts = Ref(EmceeOpts(niter, nburnin, nthin, 0.0, UInt64(seed), MODE_PHILOX, device, 0, 0, 0, 0, 0, 0, 0, 0, 0))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    create_metropolis(ld, x0, k, d, proposal, opts, h)
    s = h[]
    try
        if use_progress_meter && niter > 0                 # coarse: at most 20 polls, never per step
            done = 0
            for c in 1:min(20, niter)
                upto = (niter * c) ÷ min(20, niter)
                check(ccall((:kmc_emcee_run, LIB[]), Int32, (Ptr{Cvoid}, Int64), s, upto - done))
                done = upto
                it, m, sd, outl = Ref{Int64}(0), Ref{Float64}(0), Ref{Float64}(0), Ref{Int64}(0)
                check(ccall((:kmc_emcee_progress, LIB[]), Int32,
                    (Ptr{Cvoid}, Ref{Int64}, Ref{Float64}, Ref{Float64}, Ref{Int64}), s, it, m, sd, outl))
                nn = max(1, it[] > nburnin ? it[] - nburnin : it[])
                print(stderr, "\rmetropolis, niter=$niter, nchains=$k: $(100done ÷ niter)%  ",
                      "accept_ratio_mean=$(round(m[]/nn, sigdigits=3)) accept_ratio_std=$(round(sd[]/nn, sigdigits=3)) ",
                      "accept_ratio_outliers=$(outl[]) burnin_phase=$(it[] <= nburnin)")
            end
            println(stderr)
        else
            check(ccall((:kmc_emcee_run, LIB[]), Int32, (Ptr{Cvoid}, Int64), s, -1))
        end
        nsr = Ref{Int64}(0)
        check(ccall((:kmc_emcee_nsamples, LIB[]), Int32, (Ptr{Cvoid}, Ref{Int64}), s, nsr))
        ns = nsr[]
        th = Array{Float64,3}(undef, d, ns, k)
        lp = Matrix{Float64}(undef, ns, k)
        ar = Vector{Float64}(undef, k)
        GC.@preserve th lp ar check(ccall((:kmc_emcee_copy_results, LIB[]), Int32,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), s, th, lp, ar))
        scalar = first(starts) isa Real
        thetas = scalar ? [th[1, :, c] for c in 1:k] : [[th[:, i, c] for i in 1:ns] for c in 1:k]
        logdensities = [lp[:, c] for c in 1:k]
        nchains === nothing && return thetas[1], ar[1], logdensities[1], nothing
        return thetas, ar, logdensities, nothing
    finally
        ccall((:kmc_emcee_destroy, LIB[]), Int32, (Ptr{Cvoid},), s)
    end
end

end # module
