# b200_forwarddiff.jl — ForwardDiff support of the `:celerite_gpu` solver symbol: the body of a package extension of Pioran.jl
# (INTEGRATION.md §1, "ForwardDiff").  `logl_b200` of b200_solver.jl turns its inputs into Vector{Float64} before the `ccall`,
# so Dual numbers cannot go through it; this method catches them first.  It splits every input into values and partials,
# makes ONE pioran_celerite_logl_jvp call (B = 1, P = number of partials: ForwardDiff's chunk), and rebuilds the Dual result.
# τ never carries partials (the time stamps are data).  Any mix of Dual and Float64 inputs works: a Float64 input has zero
# tangent.  Nested Duals (Hessians) are not handled.
#
# No Julia toolchain exists in the build image of the backend: this file has not been run.  It has been checked against
# include/pioran_b200.h by hand only.

module PioranB200ForwardDiffExt

using ForwardDiff: Dual, value, partials, npartials, tagtype
import Pioran: logl_b200, logl_jvp_b200

_vals(x::AbstractVector{<:Dual}) = value.(x)
_vals(x) = x
# [length(x) × P] matrix of the partials (column p = direction p), or nothing for a Float64 input
_parts(x::AbstractVector{<:Dual}, P) = [partials(x[i], p) for i in eachindex(x), p in 1:P]
_parts(x, P) = nothing

_dualinfo(x::AbstractVector{D}) where {D <: Dual} = D
_dualinfo(x) = nothing

function logl_b200(a::AbstractVector, b::AbstractVector, c::AbstractVector, d::AbstractVector, τ, y::AbstractVector,
                   σ2::AbstractVector)
    infos = filter(!isnothing, map(_dualinfo, (a, b, c, d, y, σ2)))
    isempty(infos) && return invoke(logl_b200, Tuple{Any, Any, Any, Any, Any, Any, Any}, a, b, c, d, τ, y, σ2)
    D = first(infos)
    all(==(D), infos) || throw(ArgumentError("logl_b200: Dual inputs with different tags or chunk sizes"))
    T, P = tagtype(D), npartials(D)
    L, dL = logl_jvp_b200(_vals(a), _vals(b), _vals(c), _vals(d), τ, _vals(y), _vals(σ2),
                          _parts(a, P), _parts(b, P), _parts(c, P), _parts(d, P), _parts(y, P), _parts(σ2, P))
    return Dual{T}(L, dL...)
end

end  # module
