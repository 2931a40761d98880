# TotalLeastSquaresB200.jl -- Julia shim over libtlsq_b200.so (include/tlsq_b200.h).
#
# Drop-in replacements for the robust-PCA hot path of TotalLeastSquares.jl with the reference's own signatures,
# defaults and return types:
#     rpca(D; λ, maxrank, iters, tol, ρ, verbose, nonnegA, nonnegE, hankel, nukeA, svd, opnorm, kwargs...)
#                                   -> (A, E, s::LinearAlgebra.SVD, sv::Int)        src/robustPCA.jl:156-239
#     rpca_ga(X, r, U; verbose, tol, iters, μ) -> Q                                 src/robustPCA.jl:255-306
#     lowrankfilter(y, n; sv, lag, tol, svd, kwargs...) -> yf                       src/robustPCA.jl:119-128
#     hankel(x, L, lag) / unhankel(A, lag, N, D)                                    src/robustPCA.jl:76-92 / :28-68
#     rtls(A, y; kwargs...)                                                         src/TotalLeastSquares.jl:152-156
# Everything numerical happens behind `ccall`; this file only marshals arguments.  Julia is NOT available in the
# build image of this repository, so this shim could not be executed there: it is kept deliberately thin and the
# same C entry points are exercised by the Python mirror (totalleastsquares.jl_b200/__init__.py) in the test-suite.
#
# Usage inside TotalLeastSquares.jl (see INTEGRATION.md):
#     include("TotalLeastSquaresB200.jl"); using .TotalLeastSquaresB200
#     A, E, s, sv = TotalLeastSquaresB200.rpca(D; nonnegA = true)
module TotalLeastSquaresB200

using LinearAlgebra

export rpca, rpca_ga, lowrankfilter, hankel, unhankel, rtls, entrywise_trimmed_mean, entrywise_median

const LIB = get(ENV, "TLSQ_B200_LIB", joinpath(@__DIR__, "..", "libtlsq_b200.so"))

const TLSQ_NONNEG_A   = UInt32(1) << 0
const TLSQ_NONNEG_E   = UInt32(1) << 1
const TLSQ_HANKEL     = UInt32(1) << 2
const TLSQ_NO_NUKE_A  = UInt32(1) << 3
const TLSQ_EXACT_COST = UInt32(1) << 4

const HANDLE = Ref{Ptr{Cvoid}}(C_NULL)

function check(code::Cint)
    code == 0 && return
    msg = unsafe_string(ccall((:tlsq_last_error, LIB), Cstring, ()))
    # TLSQ_ERR_ARG (1) mirrors the reference's @assert / ArgumentError behaviour; everything else is a runtime error.
    code == 1 ? throw(ArgumentError(msg)) : error("tlsq_b200 error $code: $msg")
end

function handle()
    if HANDLE[] == C_NULL
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:tlsq_create, LIB), Cint, (Cint, Ref{Ptr{Cvoid}}), 0, h))   # no GPU => error, no CPU fallback
        HANDLE[] = h[]
    end
    HANDLE[]
end

# Element types: Float64 is native; Float32 (and integer) inputs are promoted to Float64 on the way in and the results
# converted back, so the return types match the reference's; complex inputs are not accelerated (no CPU fallback).
_check_eltype(x, name) = (eltype(x) <: Union{AbstractFloat, Integer}) ||
    throw(ArgumentError("$name: element type $(eltype(x)) is not accelerated by TotalLeastSquaresB200 (real element types only); no CPU fallback"))
_outT(x) = eltype(x) <: AbstractFloat ? eltype(x) : Float64
_back(::Type{Float64}, a) = a
_back(::Type{T}, a) where {T} = T.(a)

# ---- plugin callables (svd / opnorm kwargs, src/robustPCA.jl:168-169): the callable travels through the `user` pointer,
# the trampolines below are plain C function pointers (tlsq_svd_fn / tlsq_opnorm_fn of include/tlsq_b200.h) -------------
function _svd_tramp(user::Ptr{Cvoid}, Zp::Ptr{Float64}, M::Int64, N::Int64, sv::Int64,
                    Up::Ptr{Float64}, Sp::Ptr{Float64}, Vtp::Ptr{Float64})::Int64
    try
        f = unsafe_pointer_to_objref(user)::Base.RefValue{Any}
        s = f[][1](copy(unsafe_wrap(Array, Zp, (M, N))), Int(sv))          # svd(Z, sv)   :196
        r = min(length(s.S), M, N)
        copyto!(unsafe_wrap(Array, Up, (M, r)), @view s.U[:, 1:r])
        copyto!(unsafe_wrap(Array, Sp, (r,)), @view s.S[1:r])
        copyto!(unsafe_wrap(Array, Vtp, (r, N)), @view s.Vt[1:r, :])
        return Int64(r)
    catch err
        @error "svd callable failed" exception = err
        return Int64(-1)
    end
end
function _opnorm_tramp(user::Ptr{Cvoid}, Zp::Ptr{Float64}, M::Int64, N::Int64)::Float64
    try
        f = unsafe_pointer_to_objref(user)::Base.RefValue{Any}
        return Float64(f[][2](unsafe_wrap(Array, Zp, (M, N))))             # opnorm(Z)::RT   :177, :225
    catch err
        @error "opnorm callable failed" exception = err
        return NaN
    end
end
_is_default_svd(f) = f === LinearAlgebra.svd || f === LinearAlgebra.svd!
_is_default_opnorm(f) = f === LinearAlgebra.opnorm

"""
    A, E, s, sv = rpca(D; λ, maxrank, iters, tol, ρ, verbose, nonnegA, nonnegE, hankel, nukeA)

Same keyword list and defaults as `TotalLeastSquares.rpca` (src/robustPCA.jl:156-170); unknown keywords are swallowed
like the reference does (`kwargs...`, :170).  Non-default `svd` / `opnorm` callables (:168-169) cross the C ABI as
function pointers and run on the host (`tlsq_rpca_cb_f64`); the rest of the iteration stays on the GPU.
"""
function rpca(D::AbstractMatrix{T};
              λ              = real(T)(1.0 / sqrt(maximum(size(D)))),
              maxrank        = typemax(Int),
              iters::Int     = 1000,
              tol            = sqrt(eps(real(T))),
              ρ              = real(T)(1.5),
              verbose::Bool  = false,
              nonnegA::Bool  = false,
              nonnegE::Bool  = false,
              hankel::Bool   = false,
              nukeA          = true,
              svd::F1        = LinearAlgebra.svd!,
              opnorm::F2     = LinearAlgebra.opnorm,
              kwargs...) where {F1 <: Function, F2 <: Function, T}
    _check_eltype(D, "rpca")
    To = _outT(D)
    Dd = Matrix{Float64}(D)                         # dense, column-major (the reference copies too, :176)
    M, N = size(Dd)
    d = min(M, N)
    A, E = Matrix{Float64}(undef, M, N), Matrix{Float64}(undef, M, N)
    U, S, Vt = Matrix{Float64}(undef, M, d), Vector{Float64}(undef, d), Matrix{Float64}(undef, d, N)
    sv, its, conv = Ref{Int64}(0), Ref{Int64}(0), Ref{Int32}(0)
    hist = Matrix{Float64}(undef, 3, max(iters, 1))                  # column k = (k, svp, cost)
    flags = (nonnegA ? TLSQ_NONNEG_A : UInt32(0)) | (nonnegE ? TLSQ_NONNEG_E : UInt32(0)) |
            (hankel ? TLSQ_HANKEL : UInt32(0)) | (nukeA ? UInt32(0) : TLSQ_NO_NUKE_A) |
            (verbose ? TLSQ_EXACT_COST : UInt32(0))
    mr = maxrank == typemax(Int) ? Int64(0) : Int64(maxrank)
    if _is_default_svd(svd) && _is_default_opnorm(opnorm)
        GC.@preserve Dd A E U S Vt hist begin
            check(ccall((:tlsq_rpca_f64, LIB), Cint,
                        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Float64, Int64, Int64, Float64, Float64, UInt32,
                         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                         Ref{Int64}, Ref{Int64}, Ref{Int32}, Ptr{Float64}),
                        handle(), Dd, M, N, Float64(λ), mr, Int64(iters), Float64(tol), Float64(ρ), flags,
                        A, E, U, S, Vt, sv, its, conv, hist))
        end
    else
        # user callables: C function pointers + the callables themselves behind the opaque `user` pointer.  A NULL
        # function pointer keeps the built-in device implementation of that hook.
        box = Ref{Any}((svd, opnorm))
        svd_c = _is_default_svd(svd) ? C_NULL :
            @cfunction(_svd_tramp, Int64, (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}))
        opn_c = _is_default_opnorm(opnorm) ? C_NULL :
            @cfunction(_opnorm_tramp, Float64, (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64))
        GC.@preserve Dd A E U S Vt hist box begin
            check(ccall((:tlsq_rpca_cb_f64, LIB), Cint,
                        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Float64, Int64, Int64, Float64, Float64, UInt32,
                         Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid},
                         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                         Ref{Int64}, Ref{Int64}, Ref{Int32}, Ptr{Float64}),
                        handle(), Dd, M, N, Float64(λ), mr, Int64(iters), Float64(tol), Float64(ρ), flags,
                        svd_c, opn_c, pointer_from_objref(box),
                        A, E, U, S, Vt, sv, its, conv, hist))
        end
    end
    if verbose                                                        # :226, :229
        for k in 1:its[]
            println("$(k) cost: $(round(abs(hist[3, k]), sigdigits = 4))")
        end
        conv[] != 0 && println("converged")
    end
    conv[] == 0 && @warn "Maximum number of iterations reached, cost: $(abs(hist[3, max(its[], 1)])), tol: $tol"   # :232
    _back(To, A), _back(To, E), LinearAlgebra.SVD(_back(To, U), _back(To, S), _back(To, Vt)), Int(sv[])
end

"""
    entrywise_trimmed_mean / entrywise_median

Tags for the reference's robust averages (src/robustPCA.jl:323-333, :349-357) in `rpca_ga(...; μ = ...)`; the per-row
sorts (per-row selection beyond 16 384 observations) run on the GPU, for any number of observations.  `μ = (entrywise_trimmed_mean, P)` selects a trimming fraction other than 0.1.
"""
entrywise_trimmed_mean(args...) = error("pass it as rpca_ga(X, r; μ = entrywise_trimmed_mean)")
entrywise_median(args...) = error("pass it as rpca_ga(X, r; μ = entrywise_median)")

"""
    Q = rpca_ga(X, r = minimum(size(X)), U = similar(X); verbose = false, tol = 1e-7, iters = 1000, μ = μ!)

The start vector of every component is drawn here with `randn(d)` so the global RNG is consumed exactly like the
reference does (src/robustPCA.jl:286).  `U` is accepted for signature compatibility (the normalised copy is never
formed on the GPU).  `μ` may be `nothing` (the default weighted mean `μ!`), `entrywise_trimmed_mean`,
`(entrywise_trimmed_mean, P)` or `entrywise_median`; other callables cannot cross the C ABI.
"""
function rpca_ga(X::AbstractMatrix{T}, r = minimum(size(X)), U = nothing; verbose = false, tol = 1e-7,
                 iters::Int = 1000, μ = nothing, kwargs...) where T
    _check_eltype(X, "rpca_ga")
    To = _outT(X)
    # the averages are recognised by NAME, so the reference's own function objects (TotalLeastSquares.μ!,
    # TotalLeastSquares.entrywise_trimmed_mean, ...) select the device kernels just like the tags of this module
    fname(f) = f isa Function ? nameof(f) : :_
    kind, P = (μ === nothing || fname(μ) === :μ!) ? (0, 0.1) :
              fname(μ) === :entrywise_trimmed_mean ? (1, 0.1) :
              fname(μ) === :entrywise_median ? (2, 0.1) :
              (μ isa Tuple && fname(μ[1]) === :entrywise_trimmed_mean) ? (1, Float64(μ[2])) :
              throw(ArgumentError("rpca_ga: only μ!, entrywise_trimmed_mean and entrywise_median are supported by the B200 path"))
    Xd = Matrix{Float64}(X)
    d, N = size(Xd)
    q0 = Matrix{Float64}(undef, d, r)
    for i in 1:r
        q0[:, i] .= randn(d)                                          # :286, one draw per component, in order
    end
    Q = Matrix{Float64}(undef, d, r)
    its = Vector{Int64}(undef, r)
    GC.@preserve Xd q0 Q its begin
        check(ccall((:tlsq_rpca_ga_mu_f64, LIB), Cint,
                    (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Ptr{Float64}, Float64, Int64, Cint, Float64,
                     Ptr{Float64}, Ptr{Int64}),
                    handle(), Xd, d, N, Int64(r), q0, Float64(tol), Int64(iters), Cint(kind), P, Q, its))
    end
    verbose && foreach(i -> @info("Converged after $(its[i]) iterations"), 1:r)       # :299 (the per-iteration change of :297 stays on the device)
    any(>=(iters), its) && @warn "Reached maximum number of iterations"   # :303
    _back(To, Q)
end

"""
    yf = lowrankfilter(y, n = min(size(y,1) ÷ 20, 2000); sv = 0, lag = 1, tol = 1e-3, kwargs...)

`y` may be a vector or an `N x D` matrix of channels (src/robustPCA.jl:119-128).  One channel with `sv = 0` runs with
an implicit (never materialised) Hankel embedding; channels and the `sv > 0` plain-SSA branch (:123-125) materialise
the trajectory matrix on the device.
"""
function lowrankfilter(y::AbstractVecOrMat{T}, n = min(size(y, 1) ÷ 20, 2000); sv = 0, lag = 1, tol = 1e-3,
                       svd = LinearAlgebra.svd!, opnorm = LinearAlgebra.opnorm, λ = nothing, maxrank = typemax(Int),
                       iters::Int = 1000, ρ = 1.5, verbose::Bool = false, nonnegA::Bool = false, nonnegE::Bool = false,
                       hankel::Bool = false, nukeA = true, kwargs...) where T
    _check_eltype(y, "lowrankfilter")
    To = _outT(y)
    N, D = size(y, 1), size(y, 2)
    n <= N / 2 || throw(AssertionError("L has to be less than N/2 = $(N/2)"))       # :79
    lag <= n || throw(AssertionError("lag must be <= L"))                            # :80
    if sv <= 0 && !(_is_default_svd(svd) && _is_default_opnorm(opnorm))
        # plugin callables (test/runtests.jl:384-398): the reference's own composition (:120-127) on the materialised
        # trajectory matrix -- the callables need the whole matrix on the host anyway
        H = TotalLeastSquaresB200.hankel(Array{Float64}(y), n, lag)
        A = rpca(H; tol = tol, svd = svd, opnorm = opnorm, λ = (λ === nothing ? 1 / sqrt(maximum(size(H))) : λ),
                 maxrank = maxrank, iters = iters, ρ = ρ, verbose = verbose, nonnegA = nonnegA, nonnegE = nonnegE,
                 hankel = hankel, nukeA = nukeA)[1]
        return _back(To, unhankel(A, lag, N, D))
    end
    yd = Array{Float64}(y)
    yf = similar(yd)
    svo, its, conv = Ref{Int64}(0), Ref{Int64}(0), Ref{Int32}(0)
    flags = (nonnegA ? TLSQ_NONNEG_A : UInt32(0)) | (nonnegE ? TLSQ_NONNEG_E : UInt32(0)) |
            (hankel ? TLSQ_HANKEL : UInt32(0)) | (nukeA ? UInt32(0) : TLSQ_NO_NUKE_A)
    mr = maxrank == typemax(Int) ? Int64(0) : Int64(maxrank)
    GC.@preserve yd yf begin
        check(ccall((:tlsq_lowrankfilter_mc_f64, LIB), Cint,
                    (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Int64, Int64, Float64, Int64, Int64, Float64,
                     Float64, UInt32, Ptr{Float64}, Ref{Int64}, Ref{Int64}, Ref{Int32}, Ptr{Float64}),
                    handle(), yd, N, Int64(D), Int64(n), Int64(lag), Int64(sv), λ === nothing ? 0.0 : Float64(λ), mr,
                    Int64(iters), Float64(tol), Float64(ρ), flags, yf, svo, its, conv, C_NULL))
    end
    conv[] == 0 && @warn "Maximum number of iterations reached, tol: $tol"
    _back(To, yf)
end

"""
    X = hankel(x, L, lag = 1)          (src/robustPCA.jl:76-92; `x` is a vector or an `N x D` matrix)
"""
function hankel(x::AbstractVecOrMat{Float64}, L, lag = 1)
    N, D = size(x, 1), size(x, 2)
    K = (N - L) ÷ lag + 1
    X = Matrix{Float64}(undef, K, L * D)
    xd = Array{Float64}(x)
    GC.@preserve xd X check(ccall((:tlsq_hankel_mc_f64, LIB), Cint,
                                  (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Int64, Ptr{Float64}),
                                  handle(), xd, N, Int64(D), Int64(L), Int64(lag), X))     # asserts :79-80 -> ArgumentError
    X
end

"""
    y = unhankel(A)  /  unhankel(A, lag, N, D = 1)          (src/robustPCA.jl:28-39, 53-68)
"""
function unhankel(A::AbstractMatrix{Float64}, lag = 1, N = size(A, 2) + (size(A, 1) - 1) * lag, D = 1)
    K, L = size(A, 1), size(A, 2) ÷ D
    y = Matrix{Float64}(undef, N, D)
    Ad = Matrix{Float64}(A)
    GC.@preserve Ad y check(ccall((:tlsq_unhankel_mc_f64, LIB), Cint,
                                  (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Int64, Int64, Ptr{Float64}),
                                  handle(), Ad, K, Int64(L), Int64(lag), Int64(N), Int64(D), y))
    D == 1 ? vec(y) : y
end

"""
    x = rtls(A, y; kwargs...)          (src/TotalLeastSquares.jl:152-156: rpca([A y]; nukeA=false) then tls! on its SVD)
"""
function rtls(A::AbstractArray, y::AbstractArray; kwargs...)
    _, _, s, _ = rpca([A y]; nukeA = false, kwargs...)
    n = size(A, 2)
    V21 = s.V[1:n, n+1:end]
    V22 = s.V[n+1:end, n+1:end]
    -V21 / V22                                                       # tls!(s, n), src/TotalLeastSquares.jl:65-69
end

end # module
