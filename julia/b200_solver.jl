# b200_solver.jl — GPU backend of Pioran.jl's src/celerite_solver.jl through libpioran_b200.so (include/pioran_b200.h).
#
# Drop this file into Pioran.jl's src/ and `include("b200_solver.jl")` from src/Pioran.jl after celerite_solver.jl; then add
# the `:celerite_gpu` branch of INTEGRATION.md §2 to the three `log_likelihood` methods (src/celerite_solver.jl:262-294).
# Nothing else of the package changes: ScalableGP, approx, logpdf and the types of src/psd.jl, src/acvf.jl, src/Celerite.jl
# stay as they are.  Every `ccall` below binds one entry point of include/pioran_b200.h; tests/c_abi/abi_check.c exercises
# the same symbols from plain C and tests/test_c_abi.py pins the struct layout this file hard-codes.
#
# No Julia toolchain exists in the build image of the backend, so this file has been checked against the header by hand and
# through its C twin only (INTEGRATION.md says so too).

const libpioran_b200 = get(ENV, "PIORAN_B200_LIB", "libpioran_b200.so")

# --------------------------------------------------------------------------------------------------- context
mutable struct B200Context
    h::Ptr{Cvoid}
end
const _b200_ctx = Ref{Union{Nothing, B200Context}}(nothing)

_b200_error() = unsafe_string(ccall((:pioran_last_error, libpioran_b200), Cstring, ()))
_b200_check(rc) = rc == 0 || error("libpioran_b200 ($rc): " * _b200_error())

"""
    b200_context()

The process-wide context.  `PIORAN_B200_DEVICES="0,1,2,3"` builds ONE context over several GPUs (pioran_ctx_create_multi): a
sampler that runs as one process with one callback (examples/ultranest/single_pl.jl:113-117) then reaches every GPU of the box —
the batched entries split their parameter vectors over the devices.  Otherwise `PIORAN_B200_DEVICE` (default 0) selects one
device; under MPI, set it to `rank % ngpus` per rank.
"""
function b200_context()
    if _b200_ctx[] === nothing
        h = Ref{Ptr{Cvoid}}(C_NULL)
        if haskey(ENV, "PIORAN_B200_DEVICES")
            devs = Cint[parse(Cint, strip(s)) for s in split(ENV["PIORAN_B200_DEVICES"], ",")]
            _b200_check(ccall((:pioran_ctx_create_multi, libpioran_b200), Cint, (Ptr{Cint}, Cint, Ptr{Ptr{Cvoid}}), devs, length(devs), h))
        else
            dev = parse(Cint, get(ENV, "PIORAN_B200_DEVICE", "0"))
            _b200_check(ccall((:pioran_ctx_create, libpioran_b200), Cint, (Cint, Ptr{Ptr{Cvoid}}), dev, h))
        end
        ctx = B200Context(h[])
        finalizer(c -> ccall((:pioran_ctx_destroy, libpioran_b200), Cint, (Ptr{Cvoid},), c.h), ctx)
        _b200_ctx[] = ctx
    end
    return _b200_ctx[]
end

# --------------------------------------------------------------------------------------------------- resident series
"Resident series: (τ, y, σ²) uploaded once per sampling run (≈ 1e5 likelihood calls reuse it)."
mutable struct B200Series
    id::Cint
    N::Int
end
function b200_upload(τ::Vector{Float64}, y::Vector{Float64}, σ2::Vector{Float64})
    id = Ref{Cint}(-1)
    _b200_check(ccall((:pioran_series_upload, libpioran_b200), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        b200_context().h, length(τ), τ, y, σ2, id))
    return B200Series(id[], length(τ))
end
function b200_free(s::B200Series)
    s.id >= 0 && _b200_check(ccall((:pioran_series_free, libpioran_b200), Cint, (Ptr{Cvoid}, Cint), b200_context().h, s.id))
    s.id = -1
    return nothing
end

# Series kept on the device for the `:celerite_gpu` solver symbol, keyed by the identity of the time vector: a sampler hands
# the same `t` to every logpdf call, while `Y .- mean` and `ν .* σ²` are fresh arrays each time (src/scalable_GP.jl:162-166), so
# those two travel with the call (y_batch / s2_batch, 16 N bytes) and the series is uploaded once.
const _b200_resident = IdDict{Any, B200Series}()
function b200_resident_series(τ)
    get!(_b200_resident, τ) do
        t = collect(Float64, τ)
        b200_upload(t, zeros(length(t)), ones(length(t)))
    end
end
"Forget the resident copy of a time vector (or of all of them)."
b200_release!(τ) = haskey(_b200_resident, τ) && (b200_free(_b200_resident[τ]); delete!(_b200_resident, τ); nothing)
b200_release!() = (foreach(b200_free, values(_b200_resident)); empty!(_b200_resident); nothing)

# --------------------------------------------------------------------------------------------------- logl
"""
    logl_b200(a, b, c, d, τ, y, σ2)

Drop-in for `logl(a, b, c, d, τ, y, σ2)` (src/celerite_solver.jl:312-334), one coefficient set: the `:celerite_gpu` branch of
`log_likelihood`.  The time vector stays resident between calls (see `b200_resident_series`); y and σ² go with the call.
"""
function logl_b200(a, b, c, d, τ, y, σ2)
    out = Ref{Float64}(NaN)
    if length(τ) >= 2048
        # long series: upload (t, y, σ²) together so that the library may route the call to its parallel-in-time path
        # (pioran_ctx_set_auto_scan; per-call data arrays keep a call on the sequential sweep)
        s = b200_upload(collect(Float64, τ), collect(Float64, y), collect(Float64, σ2))
        try
            _b200_check(ccall((:pioran_celerite_logl, libpioran_b200), Cint,
                (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                 Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                b200_context().h, s.id, 1, length(a), Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
                C_NULL, C_NULL, C_NULL, C_NULL, out))
        finally
            b200_free(s)
        end
        return out[]
    end
    s = b200_resident_series(τ)
    _b200_check(ccall((:pioran_celerite_logl, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        b200_context().h, s.id, 1, length(a), Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
        C_NULL, C_NULL, collect(Float64, y), collect(Float64, σ2), out))
    return out[]
end

"""
    logl_jvp_b200(a, b, c, d, τ, y, σ2, da, db, dc, dd, dy, dσ2)

Value and P directional derivatives of `logl(a, b, c, d, τ, y, σ2)` for one coefficient set (pioran_celerite_logl_jvp with B = 1):
`da … dd` are [J × P] (column p = direction p), `dy`, `dσ2` are [N × P]; any of them may be `nothing` (zero tangent).  Returns
`(logL, dlogL::Vector{Float64})` with `dlogL[p]` the derivative along direction p.  Ranks up to 96.
"""
function logl_jvp_b200(a, b, c, d, τ, y, σ2, da, db, dc, dd, dy, dσ2)
    P = maximum(x === nothing ? 0 : size(x, 2) for x in (da, db, dc, dd, dy, dσ2))
    P >= 1 || throw(ArgumentError("logl_jvp_b200 needs at least one tangent"))
    s = b200_resident_series(τ)
    out = Ref{Float64}(NaN)
    dout = Vector{Float64}(undef, P)
    # the C ABI takes [P × J] / [P × N] row-major per parameter vector, i.e. one direction after another: Julia's column-major
    # [J × P] matrix already has that memory order
    tan(x) = x === nothing ? C_NULL : Matrix{Float64}(x)
    _b200_check(ccall((:pioran_celerite_logl_jvp, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}),
        b200_context().h, s.id, 1, length(a), P, Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
        C_NULL, C_NULL, collect(Float64, y), collect(Float64, σ2),
        tan(da), tan(db), tan(dc), tan(dd), C_NULL, C_NULL, tan(dy), tan(dσ2), out, dout))
    return out[], dout
end

"""
    logl_vjp_b200(a, b, c, d, τ, y, σ2)

Value and gradient of `logl(a, b, c, d, τ, y, σ2)` for one coefficient set from one reverse-mode sweep
(pioran_celerite_logl_vjp with B = 1).  Returns `(logL, (a = ∂a, b = ∂b, c = ∂c, d = ∂d, y = ∂y, σ2 = ∂σ2))`, each a
`Vector{Float64}` of the input's length.  A term with b = d = 0 gets ∂b = ∂d = 0 exactly.  Ranks up to 96.
"""
function logl_vjp_b200(a, b, c, d, τ, y, σ2)
    s = b200_resident_series(τ)
    J, N = length(a), length(τ)
    out = Ref{Float64}(NaN)
    ga, gb, gc, gd = (Vector{Float64}(undef, J) for _ in 1:4)
    gy, gσ2 = Vector{Float64}(undef, N), Vector{Float64}(undef, N)
    _b200_check(ccall((:pioran_celerite_logl_vjp, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}),
        b200_context().h, s.id, 1, J, Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
        C_NULL, C_NULL, collect(Float64, y), collect(Float64, σ2),
        out, ga, gb, gc, gd, C_NULL, C_NULL, gy, gσ2))
    return out[], (a = ga, b = gb, c = gc, d = gd, y = gy, σ2 = gσ2)
end

"Same against an explicitly uploaded series (its own y and σ² are used): B coefficient sets per call, rows of the [B × J] matrices."
function logl_b200(a::Matrix{Float64}, b::Matrix{Float64}, c::Matrix{Float64}, d::Matrix{Float64}, s::B200Series;
        μ::Union{Nothing, Vector{Float64}} = nothing, ν::Union{Nothing, Vector{Float64}} = nothing)
    B, J = size(a)
    out = Vector{Float64}(undef, B)
    rowmajor(m) = permutedims(m)                       # C ABI is row-major [B × J]; Julia is column-major
    _b200_check(ccall((:pioran_celerite_logl, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        b200_context().h, s.id, B, J, rowmajor(a), rowmajor(b), rowmajor(c), rowmajor(d),
        μ === nothing ? C_NULL : μ, ν === nothing ? C_NULL : ν, C_NULL, C_NULL, out))
    return out
end

# --------------------------------------------------------------------------------------------------- fused approx + logpdf
struct B200ApproxSpec   # == struct pioran_approx_spec (48 bytes; tests/test_c_abi.py pins the layout)
    psd_model::Int32
    n_components::Int32
    basis::Int32
    is_integrated_power::Int32
    f_min::Float64
    f_max::Float64
    S_low::Float64
    S_high::Float64
end

function b200_spec(psd_model::Symbol, f_min, f_max, J; basis_function = "SHO", S_low = 20.0, S_high = 20.0, is_integrated_power = true)
    model = psd_model == :SingleBendingPowerLaw ? 0 : psd_model == :DoubleBendingPowerLaw ? 1 : error("PSD model $psd_model has no fused kernel")
    basis = basis_function == "SHO" ? 0 : basis_function == "DRWCelerite" ? 1 : error("Basis function $basis_function not implemented")  # src/psd.jl:285
    return Ref(B200ApproxSpec(model, J, basis, is_integrated_power, f_min, f_max, S_low, S_high))
end

"""
    logpdf_batch(series, psd_model, Θ, f_min, f_max, J; basis_function, S_low, S_high, is_integrated_power)

Vectorised likelihood for ultranest `vectorized=true`: row i of Θ = [psd parameters…, variance, ν, μ] evaluates
logpdf(ScalableGP(μ, approx(psd_model(θ…), f_min, f_max, J, variance; basis_function))(t, ν·σ²), y)
(the body of `logl` in examples/ultranest/single_pl.jl:65-93) — approx and the celerite sweep fused on the GPU.
"""
function logpdf_batch(s::B200Series, psd_model::Symbol, Θ::Matrix{Float64}, f_min, f_max, J; kwargs...)
    spec = b200_spec(psd_model, f_min, f_max, J; kwargs...)
    B = size(Θ, 1)
    Θr = permutedims(Θ)
    out = Vector{Float64}(undef, B)
    ids = Cint[s.id]
    _b200_check(ccall((:pioran_approx_logl, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Cint}, Ptr{B200ApproxSpec}, Cint, Ptr{Float64}, Cint, Ptr{Float64}),
        b200_context().h, 1, ids, spec, B, Θr, 0, out))
    return out
end

"""
    logpdf_gradient_batch(series, psd_model, Θ, f_min, f_max, J; …) -> (logℒ::Vector, ∇::Matrix)

What `ForwardDiff.gradient(loglike, p)` returns for every row of Θ (test/test_likelihood.jl:55; the NUTS runs of
examples/turing_distributed/single_pl.jl): ∇[i, :] = ∂logℒ/∂[psd parameters…, variance, ν, μ] at Θ[i, :].
"""
function logpdf_gradient_batch(s::B200Series, psd_model::Symbol, Θ::Matrix{Float64}, f_min, f_max, J; kwargs...)
    spec = b200_spec(psd_model, f_min, f_max, J; kwargs...)
    B, P = size(Θ)
    Θr = permutedims(Θ)
    out = Vector{Float64}(undef, B)
    gr = Matrix{Float64}(undef, P, B)           # row-major [B × P] on the C side
    _b200_check(ccall((:pioran_approx_logl_grad, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Ptr{B200ApproxSpec}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        b200_context().h, s.id, spec, B, Θr, out, gr))
    return out, permutedims(gr)
end

"""
    logpdf_batch_lognormal(series, spec, Θ)

docs/src/ultranest.md:197-217 — Θ rows = [psd parameters…, variance, ν, μ, c]; upload the UNtransformed flux and σ² once: the
library computes yn = log.(y .- c), σ² = ν .* σ.^2 ./ (y .- c).^2 per row on the device.
"""
function logpdf_batch_lognormal(s::B200Series, spec::Ref{B200ApproxSpec}, Θ::Matrix{Float64})
    B = size(Θ, 1)
    Θr = permutedims(Θ)
    out = Vector{Float64}(undef, B)
    _b200_check(ccall((:pioran_approx_logl_logshift, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Ptr{B200ApproxSpec}, Cint, Ptr{Float64}, Ptr{Float64}), b200_context().h, s.id, spec, B, Θr, out))
    return out
end

# --------------------------------------------------------------------------------------------------- dense cross-check
"Drop-in for log_likelihood_direct(cov, t, y, σ²) (src/direct_solver.jl:6-21): +NLL; rethrows the reference's PosDefException."
function log_likelihood_direct_b200(a, b, c, d, t, y, σ2)
    s = b200_upload(collect(Float64, t), collect(Float64, y), collect(Float64, σ2))
    nll = Ref{Float64}(NaN)
    info = Ref{Cint}(0)
    try
        _b200_check(ccall((:pioran_direct_logl, libpioran_b200), Cint,
            (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Cint}),
            b200_context().h, s.id, 1, length(a), Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
            C_NULL, C_NULL, nll, info))
    finally
        b200_free(s)
    end
    info[] == 0 || throw(LinearAlgebra.PosDefException(info[]))
    return nll[]
end

# --------------------------------------------------------------------------------------------------- posterior mean, draws
"Drop-in for pred(a, b, c, d, τ, t, y, σ2) (src/celerite_solver.jl:376-483); τ ascending."
function pred_b200(a, b, c, d, τ, t, y, σ2)
    s = b200_upload(collect(Float64, t), collect(Float64, y), collect(Float64, σ2))
    μ = Vector{Float64}(undef, length(τ))
    try
        _b200_check(ccall((:pioran_celerite_predict, libpioran_b200), Cint,
            (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Int64, Ptr{Float64}, Ptr{Float64}),
            b200_context().h, s.id, 1, length(a), Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
            C_NULL, C_NULL, length(τ), collect(Float64, τ), μ))
    finally
        b200_free(s)
    end
    return μ
end

"""
    predict_var_b200(a, b, c, d, τ, t, y, σ2) -> (μ, v)

Posterior mean (what `pred_b200` returns, bit for bit) and variance of the latent f at ascending τ: the diagonal of
`predict_cov` (src/direct_solver.jl:28-119) in O((N + M)·R²), without measurement noise.  Ranks up to 128.
"""
function predict_var_b200(a, b, c, d, τ, t, y, σ2)
    s = b200_upload(collect(Float64, t), collect(Float64, y), collect(Float64, σ2))
    μ = Vector{Float64}(undef, length(τ))
    v = Vector{Float64}(undef, length(τ))
    try
        _b200_check(ccall((:pioran_celerite_predict_var, libpioran_b200), Cint,
            (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
            b200_context().h, s.id, 1, length(a), Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
            C_NULL, C_NULL, length(τ), collect(Float64, τ), μ, v))
    finally
        b200_free(s)
    end
    return μ, v
end

"""
    predict_cov_b200(a, b, c, d, τ, t, y, σ2) -> (μ, C)

Posterior mean (what `pred_b200` returns, bit for bit) and the M × M covariance of the latent f at ascending τ: `predict_cov`
(src/direct_solver.jl:28-119) without measurement noise, in O((N + M)·R² + M·(N + M)·R) instead of O(N³).  C is exactly
symmetric (so the row-major matrix of the C ABI reads as itself in Julia's column-major order).  Ranks up to 128.  Not run here:
no Julia toolchain.
"""
function predict_cov_b200(a, b, c, d, τ, t, y, σ2)
    s = b200_upload(collect(Float64, t), collect(Float64, y), collect(Float64, σ2))
    M = length(τ)
    μ = Vector{Float64}(undef, M)
    C = Matrix{Float64}(undef, M, M)
    try
        _b200_check(ccall((:pioran_celerite_predict_cov, libpioran_b200), Cint,
            (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
            b200_context().h, s.id, 1, length(a), Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
            C_NULL, C_NULL, M, collect(Float64, τ), μ, C))
    finally
        b200_free(s)
    end
    return μ, C
end

"""
    posterior_draws_b200(a, b, c, d, τ, t, y, σ2, q; σ2τ = 1e-18) -> Matrix (M × n)

Draws of the posterior fp(τ, σ2τ) of the zero-mean GP conditioned on (t, y, σ2), by Matheron's rule (K7): q is
`randn(rng, N + M, n)`, standard normals in the order of the merged grid of t and τ (a data point first at a tie).  O((N + M)·R)
per draw after two O((N + M)·R²) factorisations.  For the same q the draws differ from those of a dense Cholesky of
cov(fp, τ); their distribution is the same.  Ranks up to 128.  Not run here: no Julia toolchain.
"""
function posterior_draws_b200(a, b, c, d, τ, t, y, σ2, q; σ2τ = 1e-18)
    N, M = length(t), length(τ)
    size(q, 1) == N + M || throw(DimensionMismatch("q must have N + M = $(N + M) rows"))
    S = size(q, 2)
    s = b200_upload(collect(Float64, t), collect(Float64, y), collect(Float64, σ2))
    out = Matrix{Float64}(undef, M, S)   # column-major M × S is the row-major [S × M] of the C ABI
    try
        _b200_check(ccall((:pioran_celerite_posterior_draws, libpioran_b200), Cint,
            (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Int64, Ptr{Float64}, Float64, Cint, Ptr{Float64}, Ptr{Float64}),
            b200_context().h, s.id, 1, length(a), Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
            C_NULL, C_NULL, C_NULL, M, collect(Float64, τ), Float64(σ2τ), S, Matrix{Float64}(q), out))
    finally
        b200_free(s)
    end
    return out
end

"Drop-in for sim(rng, a, b, c, d, τ, σ2) (src/celerite_solver.jl:515-549): the draw q = randn(rng, N) is the reference's first line (:518)."
function sim_b200(rng, a, b, c, d, τ, σ2)
    q = randn(rng, length(τ))
    s = b200_upload(collect(Float64, τ), zeros(length(τ)), collect(Float64, σ2))
    y = Vector{Float64}(undef, length(τ))
    try
        _b200_check(ccall((:pioran_celerite_simulate, libpioran_b200), Cint,
            (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
            b200_context().h, s.id, 1, length(a), Vector{Float64}(a), Vector{Float64}(b), Vector{Float64}(c), Vector{Float64}(d),
            C_NULL, q, y))
    finally
        b200_free(s)
    end
    return y
end

"""
    sim_b200(rng, A, B, C, D, τ, σ2; ν = nothing) -> Matrix (N × P)

One draw per coefficient set: A, B, C, D are P × J (row p = the coefficients of posterior sample p), column p of the result is
`sim_b200(rng, A[p, :], B[p, :], C[p, :], D[p, :], τ, ν[p] .* σ2)` with the normals of column p of `randn(rng, N, P)`
(ν = nothing: 1).  One call for all P sets.  Not run here: no Julia toolchain.
"""
function sim_b200(rng, A::AbstractMatrix, B::AbstractMatrix, C::AbstractMatrix, D::AbstractMatrix, τ, σ2; ν = nothing)
    P, J = size(A)
    N = length(τ)
    q = randn(rng, N, P)                      # column-major N × P = row-major [P × N]
    s = b200_upload(collect(Float64, τ), zeros(N), collect(Float64, σ2))
    y = Matrix{Float64}(undef, N, P)
    row_major(X) = Matrix{Float64}(permutedims(X))   # J × P column-major = the C ABI's [P × J]
    try
        _b200_check(ccall((:pioran_celerite_simulate, libpioran_b200), Cint,
            (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
            b200_context().h, s.id, P, J, row_major(A), row_major(B), row_major(C), row_major(D),
            ν === nothing ? C_NULL : collect(Float64, ν), q, y))
    finally
        b200_free(s)
    end
    return y
end

"""
    lombscargle_b200(t, Y, dy, freq) -> Matrix (F × P)

Lomb–Scargle power of every column of Y (N × P) on the times t at the positive frequencies freq (inverse unit of t):
LombScargle.jl's `lombscargle(t, Y[:, p], dy; frequencies = freq)` with its defaults (`fit_mean`, `center_data`, `:standard`)
for every p in one call (K9).  dy = `nothing`: equal weights.  Column p of the result is the power of column p of Y.  0/0 (a
constant column, N = 1, a frequency at which the basis is degenerate on these times) gives NaN.  Not run here: no Julia toolchain.
"""
function lombscargle_b200(t, Y::AbstractVecOrMat, dy, freq)
    o = sortperm(t)                           # the power does not depend on the order of the points
    N, P = size(Y, 1), size(Y, 2)
    σ2 = dy === nothing ? ones(N) : collect(Float64, dy[o]) .^ 2
    s = b200_upload(collect(Float64, t[o]), zeros(N), σ2)
    F = length(freq)
    power = Matrix{Float64}(undef, F, P)
    try
        _b200_check(ccall((:pioran_lombscargle, libpioran_b200), Cint,
            (Ptr{Cvoid}, Cint, Cint, Ptr{Float64}, Cint, Int64, Ptr{Float64}, Ptr{Float64}),
            b200_context().h, s.id, P, Matrix{Float64}(reshape(Y, N, P)[o, :]), dy === nothing ? 0 : 1, F,
            collect(Float64, freq), power))
    finally
        b200_free(s)
    end
    return power
end

"""
    logpdf_gradient_batch_lognormal(series, spec, Θ) -> (logℒ::Vector, ∇::Matrix)

Gradient of the log-normal likelihood (docs/src/ultranest.md:197-217 under ForwardDiff): Θ rows = [psd parameters…, variance, ν, μ, c],
∇[i, :] in the same order, ∂/∂c included.
"""
function logpdf_gradient_batch_lognormal(s::B200Series, spec::Ref{B200ApproxSpec}, Θ::Matrix{Float64})
    B, P = size(Θ)
    Θr = permutedims(Θ)
    out = Vector{Float64}(undef, B)
    gr = Matrix{Float64}(undef, P, B)
    _b200_check(ccall((:pioran_approx_logl_logshift_grad, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Ptr{B200ApproxSpec}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        b200_context().h, s.id, spec, B, Θr, out, gr))
    return out, permutedims(gr)
end

"""
    logl_sine_b200(series, spec, Θ) -> Vector

The reference's periodicity run (examples/ultranest/single_pl_periodicity.jl): Θ rows = [psd parameters…, variance, ν, μ, A, ϕ, T₀],
logpdf(ScalableGP(m, approx(…))(t, ν .* σ.^2), y) with the CustomMean m(t) = μ + A·sin(2πt/T₀ + ϕ); y − A·sin(…) is formed on
the device.  Upload y and σ² once, untouched.
"""
function logl_sine_b200(s::B200Series, spec::Ref{B200ApproxSpec}, Θ::Matrix{Float64})
    B = size(Θ, 1)
    Θr = permutedims(Θ)
    out = Vector{Float64}(undef, B)
    _b200_check(ccall((:pioran_approx_logl_sine, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Ptr{B200ApproxSpec}, Cint, Ptr{Float64}, Ptr{Float64}), b200_context().h, s.id, spec, B, Θr, out))
    return out
end

"""
    logl_sine_grad_b200(series, spec, Θ) -> (logℒ::Vector, ∇::Matrix)

Gradient of `logl_sine_b200` (what ForwardDiff.gradient gives HMC/NUTS): ∇[i, :] in the column order of Θ, the partials of
A, ϕ and T₀ included.  Ranks ≤ 62.
"""
function logl_sine_grad_b200(s::B200Series, spec::Ref{B200ApproxSpec}, Θ::Matrix{Float64})
    B, P = size(Θ)
    Θr = permutedims(Θ)
    out = Vector{Float64}(undef, B)
    gr = Matrix{Float64}(undef, P, B)
    _b200_check(ccall((:pioran_approx_logl_sine_grad, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Ptr{B200ApproxSpec}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        b200_context().h, s.id, spec, B, Θr, out, gr))
    return out, permutedims(gr)
end

# --------------------------------------------------------------------------------------------------- prior transform on the device
struct B200PriorSpec   # == struct pioran_prior_spec (24 bytes)
    kind::Int32        # 0 Uniform(p0, p1) · 1 Uniform(θ[ref_col], p1) · 2 LogUniform · 3 Normal · 4 LogNormal · 5 Gamma(shape p0 ∈ ℕ, scale p1)
    ref_col::Int32     # 0-based column of the same point (kind 1)
    p0::Float64
    p1::Float64
end

"""
    prior_transform_logl_batch(series, spec, priors, cubes) -> (logℒ::Vector, Θ::Matrix)

`prior_transform` (examples/ultranest/single_pl.jl:96-104) and `logl` (:65-93) of a whole batch of unit-cube points in one call:
row i of `cubes` is mapped through the column priors (Distributions.jl quantiles) and evaluated; Θ is returned for the sampler's
bookkeeping.  For the priors of single_pl.jl:
    priors = [B200PriorSpec(0, 0, 0.0, 1.5), B200PriorSpec(2, 0, f0 * 4, fM / 4), B200PriorSpec(1, 0, 0.0, 4.0),
              B200PriorSpec(4, 0, μₙ, σₙ), B200PriorSpec(5, 0, 2.0, 0.5), B200PriorSpec(3, 0, x̄, 5 * sqrt(va))]
"""
function prior_transform_logl_batch(s::B200Series, spec::Ref{B200ApproxSpec}, priors::Vector{B200PriorSpec}, cubes::Matrix{Float64})
    B, P = size(cubes)
    cr = permutedims(cubes)
    out = Vector{Float64}(undef, B)
    Θr = Matrix{Float64}(undef, P, B)
    _b200_check(ccall((:pioran_prior_transform_logl, libpioran_b200), Cint,
        (Ptr{Cvoid}, Cint, Ptr{B200ApproxSpec}, Cint, Ptr{B200PriorSpec}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        b200_context().h, s.id, spec, P, priors, B, cr, Θr, out))
    return out, permutedims(Θr)
end
