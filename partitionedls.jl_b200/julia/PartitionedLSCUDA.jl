# PartitionedLSCUDA.jl -- thin Julia host for libpls_cuda.so (the B200 solver core).
#
# Drop-in for the bodies of
#   fit(::Type{Opt}, X, y, P; η, nnlsalg, returnAllSolutions)   PartitionedLS.jl/src/PartitionedLSOpt.jl:73-104
#   fit(::Type{BnB}, X, y, P; η, nnlsalg)                        src/PartitionedLSBnB.jl:30-40
#   fit(::Type{Alt}, X, y, P; η, ϵ, T, nnlsalg, rng)             src/PartitionedLSAlt.jl:50-124
# Everything between argument validation and the result clean-up runs in the library; `cleanupResult`
# (Opt.jl:34-44), the BnB post-processing (BnB.jl:36-39), the RNG draws of Alt (Alt.jl:58-66),
# `PartLSFitResult` (PartitionedLS.jl:29-49) and `predict` (:132-155) are the reference's own.
#
#
# The GPU solvers are selected with their own marker types -- `fit(OptCUDA, X, y, P; η)`, `fit(BnBCUDA, ...)`,
# `fit(AltCUDA, ...)` -- so this module adds methods to `PartitionedLS.fit` for types it owns: no method of the
# reference is overwritten (no type piracy; safe to precompile next to the reference, whose @compile_workload runs
# the CPU fits).  INTEGRATION.md shows the two-line change with which a maintainer routes `fit(Opt, ...)` itself
# through the library.
#
# Devices: PLS_DEVICES="0,1,2,3" (or the older single PLS_DEVICE) -- with more than one device ONE process drives
# all of them (pls_create with a device list: rows, sign patterns and restarts are sharded inside the library).
#
# NOTE: Julia is not installed in the build image, so this file has been reviewed by eye only; the
# same C ABI is exercised end to end by the Python twin (partitionedls.jl_b200/_abi.py + tests/).
module PartitionedLSCUDA

using PartitionedLS: PartLSFitResult, Opt, Alt, BnB, cleanupResult, homogeneousCoords
using Random
import PartitionedLS: fit

export OptCUDA, AltCUDA, BnBCUDA, predict_resident, fit_path

"""Marker types of the GPU solvers: `fit(OptCUDA, X, y, P; η)` is `fit(Opt, X, y, P; η)` on libpls_cuda.so."""
struct OptCUDA end
struct AltCUDA end
struct BnBCUDA end

const libpls = get(ENV, "LIBPLS_CUDA", "libpls_cuda.so")

struct PlsStats            # mirrors `pls_stats` in include/pls.h
    ms_upload::Cdouble; ms_gram::Cdouble; ms_nnls::Cdouble; ms_select::Cdouble
    ms_recompute::Cdouble; ms_total::Cdouble
    orthants::Int64; pivots::Int64; grad_evals::Int64; sum_p::Int64; sum_p2::Int64
    bpp_iters::Int64; spills::Int64; rebuilds::Int64; blocked::Int64; kernel_launches::Int64
    gram_flops::Cdouble; nnls_flops::Cdouble; nnls_l2_bytes::Cdouble
    waves::Int64; max_open::Int64; nnls_problems::Int64
    k2_variant::Int64; k2_threads::Int64; k2_ctas_per_sm::Int64; k2_grid::Int64; k2_max_drift::Cdouble
end

const _ctx = Ref{Ptr{Cvoid}}(C_NULL)      # created lazily: never ccall at precompile time
                                          # (the reference runs all fits in @compile_workload,
                                          #  PartitionedLS.jl:363-385)

function _check(rc::Cint)
    rc == 0 && return
    msg = unsafe_string(ccall((:pls_last_error, libpls), Cstring, ()))
    error("libpls_cuda: $msg (code $rc)")
end

function context()
    if _ctx[] == C_NULL
        devs = Cint[parse(Cint, strip(d)) for d in split(get(ENV, "PLS_DEVICES", get(ENV, "PLS_DEVICE", "0")), ',') if !isempty(strip(d))]
        _check(ccall((:pls_create, libpls), Cint, (Ref{Ptr{Cvoid}}, Ptr{Cint}, Cint), _ctx, devs, length(devs)))
        atexit(() -> ccall((:pls_destroy, libpls), Cvoid, (Ptr{Cvoid},), _ctx[]))
    end
    _ctx[]
end

"""
    fit(OptCUDA, X, y, P; η=0.0, nnlsalg=:nnls, returnAllSolutions=false)

Same signature and return tuple as the reference (Opt.jl:73-74, :99-103).  `nnlsalg` is accepted
and ignored: the GPU path has one Gram-space solver.  Float32 inputs are upcast (result fields are
`Vector{AbstractFloat}`, PartitionedLS.jl:34,39).
"""
function fit(::Type{OptCUDA}, X::Array{<:AbstractFloat,2}, y::AbstractArray{<:AbstractFloat,1}, P::Array{Int,2};
             η=0.0, nnlsalg=:nnls, returnAllSolutions=false)
    Xd = convert(Matrix{Float64}, X); yd = convert(Vector{Float64}, y); Pd = convert(Matrix{Int64}, P)
    N, M = size(Xd); K = size(Pd, 2)
    alpha = zeros(Float64, M + 1); b = Ref{Int64}(0); obj = Ref{Cdouble}(0.0)
    nb = 2^(K + 1)
    allobj = returnAllSolutions ? zeros(Float64, nb) : Float64[]
    allalpha = returnAllSolutions ? zeros(Float64, M + 1, nb) : zeros(Float64, 0, 0)
    stats = Ref{PlsStats}()
    GC.@preserve Xd yd Pd alpha allobj allalpha begin
        _check(ccall((:pls_opt_fit, libpls), Cint,
            (Ptr{Cvoid}, Ptr{Cdouble}, Int64, Int64, Ptr{Cdouble}, Ptr{Int64}, Int64, Cdouble, UInt32,
             Ptr{Cdouble}, Ref{Int64}, Ref{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{PlsStats}),
            context(), Xd, N, M, yd, Pd, K, Float64(η), UInt32(0),
            alpha, b, obj,
            returnAllSolutions ? pointer(allobj) : C_NULL,
            returnAllSolutions ? pointer(allalpha) : C_NULL, stats))
    end
    # the tuple of Opt.jl:92: (optval, α[1:M], β[1:K], β[K+1]*α[M+1], P), β from indextobeta (Opt.jl:4-20)
    beta(bb) = [2 * ((bb >> (k - 1)) & 1) - 1 for k in 1:K+1]
    tup(o, a, bb) = (o, a[1:end-1], beta(bb)[1:end-1], beta(bb)[end] * a[end], P)
    opt, model = cleanupResult(Opt, tup(obj[], alpha, b[]), P)
    if returnAllSolutions
        sols = [cleanupResult(Opt, tup(allobj[i], allalpha[:, i], i - 1), P) for i in 1:nb]
        return (model, nothing, (; solutions = sols))
    end
    return (model, nothing, (; opt = opt))
end

"""
    fit_path(OptCUDA, X, y, P; η::AbstractVector)

`fit(OptCUDA, X, y, P; η=η[l])` for every value of `η` (1 to 64 values, any order, duplicates allowed) on one upload
of the data (`pls_load` + `pls_opt_fit_path`): one Gram build, the orthant solves of all η, one pass over X for all
winners.  Returns a vector with one `(model, nothing, (; opt, b, stats))` per η; entry l is bitwise the model
`fit(OptCUDA, X, y, P; η=η[l])` returns (objective within 1e-12 relative).  `stats` is the call's, shared by all.
"""
function fit_path(::Type{OptCUDA}, X::Array{<:AbstractFloat,2}, y::AbstractArray{<:AbstractFloat,1}, P::Array{Int,2};
                  η::AbstractVector)
    Xd = convert(Matrix{Float64}, X); yd = convert(Vector{Float64}, y); Pd = convert(Matrix{Int64}, P)
    N, M = size(Xd); K = size(Pd, 2); L = length(η); etas = convert(Vector{Float64}, η)
    alpha = zeros(Float64, M + 1, L); b = zeros(Int64, L); obj = zeros(Float64, L); stats = Ref{PlsStats}()
    ctx = context()
    GC.@preserve Xd yd Pd etas alpha b obj begin
        _check(ccall((:pls_load, libpls), Cint,
            (Ptr{Cvoid}, Ptr{Cdouble}, Int64, Int64, Int64, Ptr{Cdouble}, Ptr{Int64}, Int64, Cdouble),
            ctx, Xd, N, N, M, yd, Pd, K, 0.0))
        _check(ccall((:pls_opt_fit_path, libpls), Cint,
            (Ptr{Cvoid}, Ptr{Cdouble}, Int64, UInt32, Ptr{Cdouble}, Ptr{Int64}, Ptr{Cdouble}, Ref{PlsStats}),
            ctx, etas, L, UInt32(0), alpha, b, obj, stats))
    end
    beta(bb) = [2 * ((bb >> (k - 1)) & 1) - 1 for k in 1:K+1]          # indextobeta, Opt.jl:4-20
    out = []
    for l in 1:L
        a = alpha[:, l]
        opt, model = cleanupResult(Opt, (obj[l], a[1:end-1], beta(b[l])[1:end-1], beta(b[l])[end] * a[end], P), P)
        push!(out, (model, nothing, (; opt = opt, b = b[l], stats = stats[])))
    end
    return out
end

"""
    fit(BnBCUDA, X, y, P; η=0.0, nnlsalg=:nnls)

Same signature and return tuple as the reference (BnB.jl:30-40).  The library returns the signed
weights α of the best feasible leaf (BnB.jl:84-89) and its objective; the post-processing of
BnB.jl:36-39 runs here unchanged.  `nopen` counts the nodes visited by the batched traversal; it
is traversal-order dependent and differs from the reference's depth-first count.
"""
function fit(::Type{BnBCUDA}, X::Array{<:AbstractFloat,2}, y::AbstractArray{<:AbstractFloat,1}, P::Array{Int,2};
             η=0.0, nnlsalg=:nnls)
    Xd = convert(Matrix{Float64}, X); yd = convert(Vector{Float64}, y); Pd = convert(Matrix{Int64}, P)
    N, M = size(Xd); K = size(Pd, 2)
    α = zeros(Float64, M + 1); obj = Ref{Cdouble}(0.0); nopen = Ref{Int64}(0); stats = Ref{PlsStats}()
    GC.@preserve Xd yd Pd α begin
        _check(ccall((:pls_bnb_fit, libpls), Cint,
            (Ptr{Cvoid}, Ptr{Cdouble}, Int64, Int64, Ptr{Cdouble}, Ptr{Int64}, Int64, Cdouble, UInt32,
             Ptr{Cdouble}, Ref{Cdouble}, Ref{Int64}, Ref{PlsStats}),
            context(), Xd, N, M, yd, Pd, K, Float64(η), UInt32(0), α, obj, nopen, stats))
    end
    _, Po = homogeneousCoords(Xd[1:1, :], Pd)            # only Po is needed (PartitionedLS.jl:76-81)
    β = sum(Po .* α, dims = 1)                           # BnB.jl:36
    α = sum(Po .* α ./ β, dims = 2)                      # BnB.jl:37 (no zero guard upstream)
    return (PartLSFitResult(α[1:end-1], β[1:end-1], β[end], P), nothing, (; opt = obj[], nopen = Int(nopen[])))
end

"""
    fit(AltCUDA, X, y, P; η=0.0, ϵ=1e-6, T=100, nnlsalg=:nnls, rng=nothing, restarts=1)

Same signature and return tuple as the reference (Alt.jl:50-51, :119) plus `restarts`: the
initial values of every restart are drawn HERE exactly as Alt.jl:58-66 does (α₀ first -- dead
upstream but it keeps the stream aligned -- then β₀ = (rng(F, K') .- 0.5) .* 10), so a given
`rng` seed means what it means upstream; the library iterates all restarts as one batch and
returns the best one.  `restarts = 1` is the reference's behaviour.
"""
function fit(::Type{AltCUDA}, X::Matrix{F}, y::Vector{F}, P::Array{Int,2};
             η=0.0, ϵ=1e-6, T=100, nnlsalg=:nnls, rng=nothing, restarts::Int=1) where {F<:AbstractFloat}
    Xd = convert(Matrix{Float64}, X); yd = convert(Vector{Float64}, y); Pd = convert(Matrix{Int64}, P)
    N, M = size(Xd); K = size(Pd, 2)
    if rng === nothing
        rng = rand
    elseif isa(rng, Int)
        Random.seed!(rng)
        rng = rand
    end
    β0 = zeros(Float64, K + 1, restarts)
    for r in 1:restarts
        rng(F, M + 1)                                    # α₀ (Alt.jl:65)
        β0[:, r] = (rng(F, K + 1) .- F(0.5)) .* 10       # β₀ (Alt.jl:66)
    end
    α = zeros(Float64, M + 1); β = zeros(Float64, K + 1); obj = Ref{Cdouble}(0.0)
    best = Ref{Int64}(0); iters = Ref{Int64}(0); stats = Ref{PlsStats}()
    GC.@preserve Xd yd Pd β0 α β begin
        _check(ccall((:pls_alt_fit, libpls), Cint,
            (Ptr{Cvoid}, Ptr{Cdouble}, Int64, Int64, Ptr{Cdouble}, Ptr{Int64}, Int64, Cdouble,
             Ptr{Cdouble}, Int64, Cdouble, Int64, UInt32,
             Ptr{Cdouble}, Ptr{Cdouble}, Ref{Cdouble}, Ref{Int64}, Ref{Int64}, Ptr{Cdouble}, Ref{PlsStats}),
            context(), Xd, N, M, yd, Pd, K, Float64(η), β0, restarts, Float64(ϵ), Int64(T), UInt32(0),
            α, β, obj, best, iters, C_NULL, stats))
    end
    return (PartLSFitResult(α[1:end-1], β[1:end-1], β[end] * α[end], P), nothing, (; opt = obj[]))   # Alt.jl:119
end

"""
    predict_resident(model, N)

`predict(model, X)` (src/PartitionedLS.jl:132-134) for the `X` of the last `fit`, which is still resident
in HBM: one streaming pass on the GPU instead of `X * (P .* α) * β .+ t` on the host.
"""
function predict_resident(model::PartLSFitResult, N::Integer)
    w = vcat(Float64.((model.P .* model.α) * model.β), Float64(model.t))
    yhat = Vector{Float64}(undef, N)
    _check(ccall((:pls_predict_resident, libpls), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), context(), w, yhat))
    return yhat
end

end # module
