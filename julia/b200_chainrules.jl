# b200_chainrules.jl — reverse-mode support of the `:celerite_gpu` solver symbol: the body of a ChainRulesCore package extension of
# Pioran.jl (INTEGRATION.md §1, "Reverse mode").  It defines `rrule(logl_b200, a, b, c, d, τ, y, σ2)`, so that every AD system that
# consumes ChainRules (Zygote, ReverseDiff through its ChainRules import, Mooncake, Enzyme through its ChainRules bridge) gets the
# gradient of the likelihood from ONE pioran_celerite_logl_vjp call (B = 1) instead of differentiating through the `ccall`.
# The pullback scales the stored gradients by the incoming cotangent; τ (the time stamps) is data and gets NoTangent().
#
# No Julia toolchain exists in the build image of the backend: this file has not been run.  It has been checked against
# include/pioran_b200.h by hand only.

module PioranB200ChainRulesExt

using ChainRulesCore: ChainRulesCore, NoTangent, unthunk
import Pioran: logl_b200, logl_vjp_b200

function ChainRulesCore.rrule(::typeof(logl_b200), a::AbstractVector, b::AbstractVector, c::AbstractVector, d::AbstractVector,
                              τ, y::AbstractVector, σ2::AbstractVector)
    L, g = logl_vjp_b200(a, b, c, d, τ, y, σ2)
    function logl_b200_pullback(ΔL)
        Δ = unthunk(ΔL)
        return (NoTangent(), Δ .* g.a, Δ .* g.b, Δ .* g.c, Δ .* g.d, NoTangent(), Δ .* g.y, Δ .* g.σ2)
    end
    return L, logl_b200_pullback
end

end  # module
