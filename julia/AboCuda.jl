# AboCuda.jl — the Julia side of the drop-in: new AbstractSurrogate / AbstractAcquisition methods
# that `ccall` into libabo_cuda.so (include/abo.h).  Written against the header; Julia is not
# available in the build image, so this file is reviewed, not executed (see INTEGRATION.md).
#
# Usage inside AbstractBayesOpt.jl (src/AbstractBayesOpt.jl:16-66): `include("AboCuda.jl")` after
# the surrogates are defined; `BOStruct` / `optimize` (src/bayesian_opt.jl:364-449) run unchanged.
module AboCuda

using LinearAlgebra
import AbstractGPs, ForwardDiff, KernelFunctions
using ..AbstractBayesOpt: AbstractSurrogate, AbstractAcquisition, ExpectedImprovement,
    ProbabilityImprovement, UpperConfidenceBound, GradientNormUCB, EnsembleAcquisition, StandardGP, GradientGP,
    extract_scale_and_lengthscale
import ..AbstractBayesOpt: update, posterior_mean, posterior_var, posterior_grad_mean, posterior_grad_var,
    posterior_grad_cov, unstandardized_mean_and_var, nlml, nlml_ls, prep_input, prep_output,
    get_lengthscale, get_scale, get_kernel_constructor, _get_minimum, _update_model_parameters,
    get_mean_std, std_y, rescale_model

const LIB = get(ENV, "ABO_CUDA_LIB", "libabo_cuda.so")
const ABO_OK, ABO_ERR_INVALID, ABO_ERR_DIM, ABO_ERR_NOT_POSDEF = 0, 1, 2, 3

last_error() = unsafe_string(ccall((:abo_last_error, LIB), Cstring, ()))
function check(rc::Int32, info::Integer=0)
    rc == ABO_OK && return nothing
    rc == ABO_ERR_NOT_POSDEF && throw(LinearAlgebra.PosDefException(info))   # caught at bayesian_opt.jl:126-141
    rc == ABO_ERR_DIM && throw(DimensionMismatch(last_error()))              # test_bayesian_opt.jl:788-817
    rc == ABO_ERR_INVALID && throw(ArgumentError(last_error()))
    error("libabo_cuda status $rc: $(last_error())")
end

mutable struct Ctx
    h::Ptr{Cvoid}
    function Ctx(device::Integer=0)
        r = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:abo_ctx_create, LIB), Int32, (Int32, Ref{Ptr{Cvoid}}), device, r))
        c = new(r[]); finalizer(c -> ccall((:abo_ctx_destroy, LIB), Int32, (Ptr{Cvoid},), c.h), c); c
    end
end
const DEFAULT_CTX = Ref{Union{Nothing,Ctx}}(nothing)
ctx() = (DEFAULT_CTX[] === nothing && (DEFAULT_CTX[] = Ctx(0)); DEFAULT_CTX[])

mutable struct Handle            # abo_gp*: a conditioned surrogate resident in HBM
    h::Ptr{Cvoid}
    Handle(h) = (x = new(h); finalizer(x -> ccall((:abo_gp_destroy, LIB), Int32, (Ptr{Cvoid},), x.h), x); x)
end

const KERNEL_IDS = Dict(:SqExponentialKernel => 0, :Matern52Kernel => 1, :Matern72Kernel => 2,
    :ApproxMatern52Kernel => 3, :ApproxMatern72Kernel => 4, :ADMatern52Kernel => 5, :ADMatern72Kernel => 6)

# hyper-parameters of a handle: ScaleTransform (one stored s = 1/l, SURVEY H4) or ARDTransform (one per dimension — not
# constructible through the reference's constructors today, src/bayesian_opt.jl:193-194 lists it as a TODO, but a kernel
# built by hand with `base ∘ ARDTransform(1 ./ l)` is honoured by every device path)
function set_params!(h, transform, scale::Float64, noise::Float64, mc::Vector{Float64})
    if transform isa KernelFunctions.ARDTransform
        v = collect(Float64, transform.v)
        check(GC.@preserve v mc ccall((:abo_gp_set_params_ard, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Float64, Float64, Ptr{Float64}),
            h.h, v, scale, noise, mc))
    else
        check(GC.@preserve mc ccall((:abo_gp_set_params, LIB), Int32, (Ptr{Cvoid}, Float64, Float64, Float64, Ptr{Float64}),
            h.h, Float64(transform.s[1]), scale, noise, mc))
    end
end

"""GPU twin of StandardGP (src/surrogates/StandardGP.jl:11-16): same prior description, the posterior
is a device handle instead of an AbstractGPs.PosteriorGP."""
struct CuStandardGP{T} <: AbstractSurrogate
    prior::StandardGP{T}              # keeps kernel / noise / mean exactly as the reference stores them
    gpx::Union{Nothing,Handle}
    X::Union{Nothing,Matrix{Float64}} # conditioning data (d x n) the handle holds: enables the O(n^2) append
    y::Union{Nothing,Vector{Float64}}
end
CuStandardGP(prior::StandardGP, gpx) = CuStandardGP(prior, gpx, nothing, nothing)
CuStandardGP(kernel, noise_var; mean=nothing) = CuStandardGP(StandardGP(kernel, noise_var; mean=mean), nothing)

get_lengthscale(m::CuStandardGP) = get_lengthscale(m.prior)
get_scale(m::CuStandardGP) = get_scale(m.prior)
get_kernel_constructor(m::CuStandardGP) = get_kernel_constructor(m.prior)
prep_input(m::CuStandardGP, xs) = xs
prep_output(m::CuStandardGP, ys) = ys
_get_minimum(m::CuStandardGP, ys) = minimum(ys)
get_mean_std(m::CuStandardGP, ys, choice) = get_mean_std(m.prior, ys, choice)
std_y(m::CuStandardGP, ys, μ, σ) = std_y(m.prior, ys, μ, σ)
rescale_model(m::CuStandardGP, σ) = CuStandardGP(rescale_model(m.prior, σ), nothing)
_update_model_parameters(m::CuStandardGP, k) = CuStandardGP(_update_model_parameters(m.prior, k), nothing)

transform_of(m::CuStandardGP) = m.prior.gp.kernel.kernel.transform
kernel_id(m::CuStandardGP) = KERNEL_IDS[nameof(typeof(get_kernel_constructor(m)))]
inv_lengthscale(m::CuStandardGP) = m.prior.gp.kernel.kernel.transform.s[1]   # the stored s, not 1/ℓ (SURVEY H4)
mean_const(m::CuStandardGP) = m.prior.gp.mean isa AbstractGPs.ZeroMean ? 0.0 : m.prior.gp.mean.c

function Base.copy(m::CuStandardGP)                                           # StandardGP.jl:26
    m.gpx === nothing && return CuStandardGP(m.prior, nothing)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:abo_gp_clone, LIB), Int32, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}), m.gpx.h, r))
    CuStandardGP(m.prior, Handle(r[]), m.X, m.y)      # O(1): the clone shares the device buffers (copy-on-write)
end

points(xs::Vector{<:AbstractVector}) = reduce(hcat, xs)                       # d x n column-major = point-major
points(xs::Vector{<:Real}) = reshape(collect(Float64, xs), 1, :)

function update(m::CuStandardGP, xs::Vector, ys::Vector)                      # StandardGP.jl:79-83
    X = Matrix{Float64}(points(xs)); d, n = size(X)
    length(ys) == n || throw(DimensionMismatch("xs and ys have different lengths"))
    y = collect(Float64, ys)
    # one more observation on top of what the handle already holds (the BO loop, bayesian_opt.jl:120-125):
    # O(n^2) row append on a copy-on-write clone instead of the O(n^3) re-fit
    if m.gpx !== nothing && m.X !== nothing && size(m.X, 2) == n - 1 && size(m.X, 1) == d &&
       view(X, :, 1:n-1) == m.X && view(y, 1:n-1) == m.y
        c = copy(m); info = Ref{Int64}(0)
        xn = X[:, n]; yn = [y[n]]
        rc = GC.@preserve xn yn ccall((:abo_gp_append, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ref{Int64}),
            c.gpx.h, xn, yn, info)
        check(rc, info[])
        return CuStandardGP(m.prior, c.gpx, X, y)
    end
    r = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:abo_gp_create, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ref{Ptr{Cvoid}}),
        ctx().h, kernel_id(m), d, 1, r))
    h = Handle(r[])
    mc = [Float64(mean_const(m))]
    set_params!(h, transform_of(m), Float64(get_scale(m)[1]), Float64(m.prior.noise_var), mc)
    info = Ref{Int64}(0)
    rc = GC.@preserve X y ccall((:abo_gp_fit, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ref{Int64}),
        h.h, X, y, n, info)
    check(rc, info[])
    CuStandardGP(m.prior, h, X, y)
end

function posterior(m::CuStandardGP, x::AbstractVector, want_mean::Bool, want_var::Bool)
    Xc = Matrix{Float64}(points(collect(x))); mcount = size(Xc, 2)
    μ = want_mean ? Vector{Float64}(undef, mcount) : Float64[]
    v = want_var ? Vector{Float64}(undef, mcount) : Float64[]
    check(GC.@preserve Xc μ v ccall((:abo_gp_posterior, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ptr{Float64}, Ptr{Float64}),
        m.gpx.h, Xc, mcount, 1, want_mean ? pointer(μ) : C_NULL, want_var ? pointer(v) : C_NULL))
    μ, v
end
posterior_mean(m::CuStandardGP, x::AbstractVector) = posterior(m, x, true, false)[1]   # StandardGP.jl:361-363
posterior_var(m::CuStandardGP, x::AbstractVector) = posterior(m, x, false, true)[2]    # StandardGP.jl:377-379
posterior_mean(m::CuStandardGP, x::Real) = posterior_mean(m, [x])
posterior_var(m::CuStandardGP, x::Real) = posterior_var(m, [x])

# ---- fused acquisitions: one sweep instead of two posterior passes (ExpectedImprovement.jl:40-45)
acq_id(::ExpectedImprovement) = Int32(0); acq_params(a::ExpectedImprovement) = Float64[a.ξ, a.best_y]
acq_id(::ProbabilityImprovement) = Int32(1); acq_params(a::ProbabilityImprovement) = Float64[a.ξ, a.best_y]
acq_id(::UpperConfidenceBound) = Int32(2); acq_params(a::UpperConfidenceBound) = Float64[a.β]

function acq_eval(a::AbstractAcquisition, m::CuStandardGP, x::AbstractVector; k::Integer=0)
    Xc = Matrix{Float64}(points(collect(x))); mcount = size(Xc, 2)
    scores = Vector{Float64}(undef, mcount); p = acq_params(a)
    ti = Vector{Int64}(undef, max(k, 1)); tv = Vector{Float64}(undef, max(k, 1))
    check(GC.@preserve Xc scores p ti tv ccall((:abo_acq_eval, LIB), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Float64}),
        m.gpx.h, acq_id(a), p, Xc, mcount, scores, min(k, mcount), ti, tv))
    scores, ti[1:min(k, mcount)] .+ 1, tv[1:min(k, mcount)]        # 0-based -> Julia indices
end
(a::ExpectedImprovement)(m::CuStandardGP, x::AbstractVector) = acq_eval(a, m, x)[1]
(a::ProbabilityImprovement)(m::CuStandardGP, x::AbstractVector) = acq_eval(a, m, x)[1]
(a::UpperConfidenceBound)(m::CuStandardGP, x::AbstractVector) = acq_eval(a, m, x)[1]

# acquisition value and its analytic gradient for a batch of points in one call: what a batched replacement of
# the finite-difference refinement loop (acq_utils.jl:55-71) evaluates per step
function acq_value_grad(a::AbstractAcquisition, m::CuStandardGP, x::AbstractVector)
    Xc = Matrix{Float64}(points(collect(x))); d, mcount = size(Xc)
    scores = Vector{Float64}(undef, mcount); grad = Matrix{Float64}(undef, d, mcount); p = acq_params(a)
    check(GC.@preserve Xc scores grad p ccall((:abo_acq_eval_grad, LIB), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        m.gpx.h, acq_id(a), p, Xc, mcount, scores, grad, C_NULL, C_NULL))
    scores, grad                                                   # grad[:, c] = d acq / d x_c
end

# ---- nlml with ForwardDiff.Dual parameters (bayesian_opt.jl:284): value + analytic gradient from the
#      device, re-assembled into a Dual (SURVEY H7)
function nlml_value_grad(m::CuStandardGP, θ::Vector{Float64}, xs, ys)
    X = Matrix{Float64}(points(xs)); d, n = size(X); y = collect(Float64, ys)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:abo_gp_create, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ref{Ptr{Cvoid}}), ctx().h, kernel_id(m), d, 1, r))
    h = Handle(r[]); mc = [Float64(mean_const(m))]
    set_params!(h, transform_of(m), Float64(get_scale(m)[1]), Float64(m.prior.noise_var), mc)
    val = Ref{Float64}(0.0); g = zeros(2); info = Ref{Int32}(0)
    check(GC.@preserve X y θ g ccall((:abo_nlml_batch, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ref{Float64}, Ptr{Float64}, Ref{Int32}),
        h.h, X, y, n, θ, 1, val, g, info))
    info[] != 0 && throw(LinearAlgebra.PosDefException(info[]))
    val[], g
end
nlml(m::CuStandardGP, p::AbstractVector{<:AbstractFloat}, xs, ys) = nlml_value_grad(m, collect(Float64, p), xs, ys)[1]
function nlml(m::CuStandardGP, p::AbstractVector{D}, xs, ys) where {T,V,N,D<:ForwardDiff.Dual{T,V,N}}
    v, g = nlml_value_grad(m, Float64.(ForwardDiff.value.(p)), xs, ys)
    parts = g[1] * ForwardDiff.partials(p[1]) + g[2] * ForwardDiff.partials(p[2])
    ForwardDiff.Dual{T}(v, parts)
end
nlml_ls(m::CuStandardGP, log_ℓ, log_scale::Float64, xs, ys) = nlml(m, [log_ℓ, oftype(log_ℓ, log_scale)], xs, ys)


# unstandardized_mean_and_var(::StandardGP, xs, params) (StandardGP.jl:395-404; tutorials 2D_BO.jl:177): mean and variance
# from ONE sweep instead of mean_and_var on a FiniteGP
function unstandardized_mean_and_var(m::CuStandardGP, xs::AbstractVector, params)
    μ, σ = params
    mn, v = posterior(m, xs, true, true)
    (mn .* σ) .+ μ, v .* (σ^2)
end

# =====================================================================================================================
# CuGradientGP — GPU twin of GradientGP (src/surrogates/GradientGP.jl:17-22): value + gradient observations, the
# N = n (d + 1) system with the derivative blocks of gradKernel (:573-606) built, factorised and queried on the device.
# Observations cross the ABI OUT-MAJOR, exactly prep_output (:919-922); multi-output results come back out-major.
# =====================================================================================================================
struct CuGradientGP{T} <: AbstractSurrogate
    prior::GradientGP{T}
    gpx::Union{Nothing,Handle}
    X::Union{Nothing,Matrix{Float64}}   # d x n conditioning points held by the handle
    y::Union{Nothing,Vector{Float64}}   # out-major observations (length n p)
end
CuGradientGP(prior::GradientGP, gpx) = CuGradientGP(prior, gpx, nothing, nothing)
CuGradientGP(kernel, p::Int, noise_var; kw...) = CuGradientGP(GradientGP(kernel, p, noise_var; kw...), nothing)

get_lengthscale(m::CuGradientGP) = get_lengthscale(m.prior)
get_scale(m::CuGradientGP) = get_scale(m.prior)
get_kernel_constructor(m::CuGradientGP) = get_kernel_constructor(m.prior)
prep_input(m::CuGradientGP, xs) = xs                                   # the device builds the multi-output layout itself
prep_output(m::CuGradientGP, ys::Vector) = prep_output(m.prior, ys)    # vec(permutedims(hcat(ys...))): out-major
_get_minimum(m::CuGradientGP, ys) = _get_minimum(m.prior, ys)
get_mean_std(m::CuGradientGP, ys, choice) = get_mean_std(m.prior, ys, choice)
std_y(m::CuGradientGP, ys, μ, σ) = std_y(m.prior, ys, μ, σ)
rescale_model(m::CuGradientGP, σ) = CuGradientGP(rescale_model(m.prior, σ), nothing)
_update_model_parameters(m::CuGradientGP, k) = CuGradientGP(_update_model_parameters(m.prior, k), nothing)

transform_of(m::CuGradientGP) = m.prior.gp.kernel.base_kernel.kernel.transform
kernel_id(m::CuGradientGP) = KERNEL_IDS[nameof(typeof(get_kernel_constructor(m)))]
inv_lengthscale(m::CuGradientGP) = m.prior.gp.kernel.base_kernel.kernel.transform.s[1]   # stored s (GradientGP.jl:842)
# gradConstMean's constructor returns a CustomMean closing over c (GradientGP.jl:505-515): evaluate it per output
mean_consts(m::CuGradientGP, x1) = Float64[AbstractGPs.mean_vector(m.prior.gp.mean, [(x1, o)])[1] for o in 1:m.prior.p]

function Base.copy(m::CuGradientGP)                                    # GradientGP.jl:32
    m.gpx === nothing && return CuGradientGP(m.prior, nothing)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:abo_gp_clone, LIB), Int32, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}), m.gpx.h, r))
    CuGradientGP(m.prior, Handle(r[]), m.X, m.y)
end

function update(m::CuGradientGP, xs::AbstractVector, ys::AbstractVector)   # GradientGP.jl:659-668
    X = Matrix{Float64}(points(collect(xs))); d, n = size(X); p = m.prior.p
    p == d + 1 || throw(DimensionMismatch("GradientGP: p must equal d + 1"))
    (length(ys) == n && all(length(y) == p for y in ys)) || throw(DimensionMismatch("ys must hold n vectors of length p"))
    y = collect(Float64, vec(permutedims(reduce(hcat, ys))))           # out-major: [f(x1..xn); d1 f(x1..xn); ...]
    # one more point on top of what the handle holds: block append of its p rows, O(N^2 p), on a copy-on-write clone
    if m.gpx !== nothing && m.X !== nothing && size(m.X) == (d, n - 1) && view(X, :, 1:n-1) == m.X &&
       reshape(y, n, p)[1:n-1, :] == reshape(m.y, n - 1, p)
        c = copy(m); info = Ref{Int64}(0)
        xn = X[:, n]; yn = collect(Float64, ys[n])
        rc = GC.@preserve xn yn ccall((:abo_gp_append, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ref{Int64}),
            c.gpx.h, xn, yn, info)
        check(rc, info[])
        return CuGradientGP(m.prior, c.gpx, X, y)
    end
    r = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:abo_gp_create, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ref{Ptr{Cvoid}}),
        ctx().h, kernel_id(m), d, p, r))
    h = Handle(r[])
    mc = mean_consts(m, X[:, 1])
    set_params!(h, transform_of(m), Float64(get_scale(m)[1]), Float64(m.prior.noise_var), mc)
    info = Ref{Int64}(0)
    rc = GC.@preserve X y ccall((:abo_gp_fit, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ref{Int64}),
        h.h, X, y, n, info)
    check(rc, info[])
    CuGradientGP(m.prior, h, X, y)
end

# outputs = 1: value only (posterior_mean / posterior_var, GradientGP.jl:985-1003); outputs = p: all outputs, out-major
function posterior(m::CuGradientGP, x::AbstractVector, outputs::Integer, want_mean::Bool, want_var::Bool)
    Xc = Matrix{Float64}(points(collect(x))); mcount = size(Xc, 2)
    μ = want_mean ? Vector{Float64}(undef, mcount * outputs) : Float64[]
    v = want_var ? Vector{Float64}(undef, mcount * outputs) : Float64[]
    check(GC.@preserve Xc μ v ccall((:abo_gp_posterior, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ptr{Float64}, Ptr{Float64}),
        m.gpx.h, Xc, mcount, outputs, want_mean ? pointer(μ) : C_NULL, want_var ? pointer(v) : C_NULL))
    μ, v
end
posterior_mean(m::CuGradientGP, x::AbstractVector) = posterior(m, x, 1, true, false)[1]
posterior_var(m::CuGradientGP, x::AbstractVector) = posterior(m, x, 1, false, true)[2]
posterior_mean(m::CuGradientGP, x::Real) = posterior_mean(m, [x])
posterior_var(m::CuGradientGP, x::Real) = posterior_var(m, [x])
posterior_grad_mean(m::CuGradientGP, x) = posterior(m, x, m.prior.p, true, false)[1]     # GradientGP.jl:936-939
posterior_grad_var(m::CuGradientGP, x) = posterior(m, x, m.prior.p, false, true)[2]      # GradientGP.jl:952-955
function posterior_grad_cov(m::CuGradientGP, x)                                          # GradientGP.jl:968-971
    Xc = Matrix{Float64}(points(collect(x))); mcount = size(Xc, 2); M = mcount * m.prior.p
    cov = Matrix{Float64}(undef, M, M)
    check(GC.@preserve Xc cov ccall((:abo_gp_posterior_cov, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ptr{Float64}), m.gpx.h, Xc, mcount, m.prior.p, cov))
    cov                                                                # symmetric: row- vs column-major is immaterial
end

function unstandardized_mean_and_var(m::CuGradientGP, X, params::Tuple)                  # GradientGP.jl:1019-1030
    μ, σ = params[1], params[2][1]
    mn, v = posterior(m, X, m.prior.p, true, true)
    (reshape(mn, :, m.prior.p) .* σ) .+ μ', reshape(v, :, m.prior.p) .* (σ^2)
end

# value-output acquisitions on a GradientGP: the same fused sweep (K* has value and derivative rows, value column only)
function acq_eval(a::AbstractAcquisition, m::CuGradientGP, x::AbstractVector; k::Integer=0)
    Xc = Matrix{Float64}(points(collect(x))); mcount = size(Xc, 2)
    scores = Vector{Float64}(undef, mcount); p = acq_params(a)
    ti = Vector{Int64}(undef, max(k, 1)); tv = Vector{Float64}(undef, max(k, 1))
    check(GC.@preserve Xc scores p ti tv ccall((:abo_acq_eval, LIB), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Float64}),
        m.gpx.h, acq_id(a), p, Xc, mcount, scores, min(k, mcount), ti, tv))
    scores, ti[1:min(k, mcount)] .+ 1, tv[1:min(k, mcount)]
end
(a::ExpectedImprovement)(m::CuGradientGP, x::AbstractVector) = acq_eval(a, m, x)[1]
(a::ProbabilityImprovement)(m::CuGradientGP, x::AbstractVector) = acq_eval(a, m, x)[1]
(a::UpperConfidenceBound)(m::CuGradientGP, x::AbstractVector) = acq_eval(a, m, x)[1]

# GradientNormUCB (gradNormUCB.jl:43-51) and EnsembleAcquisition (EnsembleAcq.jl:53-55): all members from ONE posterior
# pass on the device; the reference calls posterior_grad_mean + posterior_grad_cov once per candidate and per member
acq_id(::GradientNormUCB) = Int32(3); acq_params(a::GradientNormUCB) = Float64[a.β, 0.0]
member_params(a) = (p = acq_params(a); length(p) == 2 ? p : Float64[p[1], 0.0])
function acq_eval_multi(members::Vector, weights::Vector{Float64}, m::Union{CuStandardGP,CuGradientGP}, x::AbstractVector; k::Integer=0)
    Xc = Matrix{Float64}(points(collect(x))); mcount = size(Xc, 2); nm = length(members)
    ids = Int32[acq_id(a) for a in members]
    pars = reduce(hcat, [member_params(a) for a in members])          # 2 x nmem column-major = nmem x 2 row-major
    scores = Vector{Float64}(undef, mcount)
    ti = Vector{Int64}(undef, max(k, 1)); tv = Vector{Float64}(undef, max(k, 1))
    check(GC.@preserve Xc ids weights pars scores ti tv ccall((:abo_acq_eval_multi, LIB), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Float64}),
        m.gpx.h, nm, ids, weights, pars, Xc, mcount, scores, min(k, mcount), ti, tv))
    scores, ti[1:min(k, mcount)] .+ 1, tv[1:min(k, mcount)]
end
(a::GradientNormUCB)(m::CuGradientGP, x::AbstractVector) = acq_eval_multi(Any[a], [1.0], m, x)[1]
const FusableAcq = Union{ExpectedImprovement,ProbabilityImprovement,UpperConfidenceBound,GradientNormUCB}
function (ea::EnsembleAcquisition)(m::Union{CuStandardGP,CuGradientGP}, x::AbstractVector)
    if all(a -> a isa FusableAcq, ea.acquisitions) && length(ea.acquisitions) <= 8
        return acq_eval_multi(collect(Any, ea.acquisitions), collect(Float64, ea.weights), m, x)[1]
    end
    sum([ea.weights[i] .* ea.acquisitions[i](m, x) for i in eachindex(ea.weights)])      # EnsembleAcq.jl:53-55
end

# nlml(::GradientGP, params, xs, ys) (GradientGP.jl:684-738) incl. ForwardDiff.Dual parameters: xs / ys arrive already
# prepared by optimize_hyperparameters (prep_input / prep_output, bayesian_opt.jl:250-251): xs the plain points,
# ys the out-major vector
function nlml_value_grad(m::CuGradientGP, θ::Vector{Float64}, xs, ys)
    X = Matrix{Float64}(points(collect(xs))); d, n = size(X); p = m.prior.p
    y = ys isa AbstractVector{<:Real} ? collect(Float64, ys) : collect(Float64, vec(permutedims(reduce(hcat, ys))))
    length(y) == n * p || throw(DimensionMismatch("ys must hold n p values"))
    r = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:abo_gp_create, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ref{Ptr{Cvoid}}), ctx().h, kernel_id(m), d, p, r))
    h = Handle(r[]); mc = mean_consts(m, X[:, 1])
    set_params!(h, transform_of(m), Float64(get_scale(m)[1]), Float64(m.prior.noise_var), mc)
    val = Ref{Float64}(0.0); g = zeros(2); info = Ref{Int32}(0)
    check(GC.@preserve X y θ g ccall((:abo_nlml_batch, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ref{Float64}, Ptr{Float64}, Ref{Int32}),
        h.h, X, y, n, θ, 1, val, g, info))
    info[] != 0 && throw(LinearAlgebra.PosDefException(info[]))
    val[], g
end
nlml(m::CuGradientGP, p::AbstractVector{<:AbstractFloat}, xs, ys) = nlml_value_grad(m, collect(Float64, p), xs, ys)[1]
function nlml(m::CuGradientGP, p::AbstractVector{D}, xs, ys) where {T,V,N,D<:ForwardDiff.Dual{T,V,N}}
    v, g = nlml_value_grad(m, Float64.(ForwardDiff.value.(p)), xs, ys)
    ForwardDiff.Dual{T}(v, g[1] * ForwardDiff.partials(p[1]) + g[2] * ForwardDiff.partials(p[2]))
end
nlml_ls(m::CuGradientGP, log_ℓ, log_scale::Float64, xs, ys) = nlml(m, [log_ℓ, oftype(log_ℓ, log_scale)], xs, ys)

# get_mean_std + std_y of standardize_problem (src/BO_utils.jl:44-64) in one device call: (μ, σ, standardised ys, incumbent).
# `ys` as the BO loop holds them (Vector{Float64} or Vector{Vector{Float64}}); returns ys in the same shape.
const STD_CHOICE = Dict("mean_scale" => Int32(0), "scale_only" => Int32(1), "mean_only" => Int32(2))
function standardize_device(m::Union{CuStandardGP,CuGradientGP}, ys::AbstractVector, choice::String)
    grad = m isa CuGradientGP
    p = grad ? m.prior.p : 1; n = length(ys)
    y = grad ? collect(Float64, vec(permutedims(reduce(hcat, ys)))) : collect(Float64, ys)    # out-major
    μ = Vector{Float64}(undef, p); σ = Vector{Float64}(undef, p); ystd = similar(y); best = Ref{Float64}(0.0)
    check(GC.@preserve y μ σ ystd ccall((:abo_standardize, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Float64}),
        ctx().h, y, n, p, STD_CHOICE[choice], μ, σ, ystd, best))
    grad ? (μ, σ, [collect(r) for r in eachrow(reshape(ystd, n, p))], best[]) : (μ[1], σ[1], ystd, best[])
end

# ARD marginal likelihood: θ = (log l_1 .. log l_d, log σ²), value and analytic gradient (d + 1) in one call — the extension
# of the nlml parameter vector planned at src/bayesian_opt.jl:193-194
function nlml_ard_value_grad(m::CuStandardGP, θ::Vector{Float64}, xs, ys)
    X = Matrix{Float64}(points(xs)); d, n = size(X); y = collect(Float64, ys)
    length(θ) == d + 1 || throw(DimensionMismatch("θ must hold d + 1 entries"))
    r = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:abo_gp_create, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, Ref{Ptr{Cvoid}}), ctx().h, kernel_id(m), d, 1, r))
    h = Handle(r[]); mc = [Float64(mean_const(m))]
    set_params!(h, transform_of(m), Float64(get_scale(m)[1]), Float64(m.prior.noise_var), mc)
    val = Ref{Float64}(0.0); g = zeros(d + 1); info = Ref{Int32}(0)
    check(GC.@preserve X y θ g ccall((:abo_nlml_batch_ard, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ref{Float64}, Ptr{Float64}, Ref{Int32}),
        h.h, X, y, n, θ, 1, val, g, info))
    info[] != 0 && throw(LinearAlgebra.PosDefException(info[]))
    val[], g
end

# Joint draws of the latent value over xs, AbstractGPs rand(rng, posterior(fx)(xs), S): an m x S matrix, column s = draw s
# (the library's sample-major S x m buffer is exactly this matrix in column-major order).  Draw s depends only on
# (seed, s); jitter is relative to the kernel scale and raised tenfold, up to six times, until the covariance factors.
# Thompson sampling proposes argmin of each column (argmin(posterior_sample(m, xs, q; seed=seed), dims=1)).
function posterior_sample(m::Union{CuStandardGP,CuGradientGP}, xs, S::Integer; seed::Integer, jitter::Real=1e-10)
    m.gpx === nothing && error("surrogate has no posterior: call update(model, xs, ys) first")
    Xc = Matrix{Float64}(points(collect(xs))); mcount = size(Xc, 2)
    out = Matrix{Float64}(undef, mcount, S)
    τ = Ref{Float64}(0.0)
    check(GC.@preserve Xc out ccall((:abo_gp_posterior_sample, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, UInt64, Float64, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ref{Float64}),
        m.gpx.h, Xc, mcount, S, UInt64(seed), Float64(jitter), out, C_NULL, C_NULL, τ))
    out
end

# monte_carlo_fill_distance (src/BO_utils.jl:140-159) on the device; the caller draws the uniform samples
function fill_distance(X::Matrix{Float64}, S::Matrix{Float64})         # both d x count, column-major = point-major
    out = Ref{Float64}(0.0)
    check(GC.@preserve X S ccall((:abo_fill_distance, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ptr{Float64}, Int64, Ref{Float64}),
        ctx().h, X, size(X, 2), size(X, 1), S, size(S, 2), out))
    out[]
end

end # module
