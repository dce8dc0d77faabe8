/*
 * pioran_b200.h — C ABI of libpioran_b200.so, the B200 (sm_100a) backend of Pioran.jl's likelihood hot path.
 *
 * The reference (mlefkir/Pioran.jl, pure Julia) has no FFI of its own; its operator boundary for this path is
 * Julia dispatch on  log_likelihood(cov, τ, y, σ2; solver::Symbol)  (src/celerite_solver.jl:262-294), selected by
 * the `solver` field of ScalableGP (src/scalable_GP.jl:24-40,162-166).  Each entry point below names the reference
 * function it stands in for; INTEGRATION.md shows the `ccall` stubs a Pioran maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / CUDA types in any signature (streams are passed as void*).
 *   - every function returns 0 on success or a negative PIORAN_E* code; it never throws or aborts.
 *     pioran_last_error() returns a thread-local, NUL-terminated description of the last failure.
 *   - logL values that are NaN/±Inf are data (a non-positive-definite θ), not errors — like the reference, which
 *     takes log|D_n| (src/celerite_solver.jl:140) and never checks definiteness on the celerite path.
 *   - pointers are HOST memory unless the function name ends in `_dev`; the caller owns every buffer and the
 *     library keeps no pointer after return.  A context is bound to one CUDA device; one context per thread.
 *   - all floating point is IEEE double (FP64); there is no CPU fallback: with no usable GPU every call fails
 *     with PIORAN_ECUDA.
 */
#ifndef PIORAN_B200_H
#define PIORAN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIORAN_OK 0
#define PIORAN_EINVAL (-1)  /* bad argument (message in pioran_last_error)            */
#define PIORAN_ECUDA (-2)   /* CUDA runtime / driver failure, or no sm_100 device     */
#define PIORAN_ENOMEM (-3)  /* host or device allocation failed                       */
#define PIORAN_ESINGULAR (-4) /* spectral matrix of approx() is singular              */
#define PIORAN_EUNSUPPORTED (-5) /* shape outside the compiled kernel set             */

/* Tonari.jl PSD models usable on the fused path (formulas pinned by reference test/test_psd.jl:6,12). */
#define PIORAN_PSD_SBPL 0 /* SingleBendingPowerLaw(α₁, f₁, α₂)            — 3 parameters */
#define PIORAN_PSD_DBPL 1 /* DoubleBendingPowerLaw(α₁, f₁, α₂, f₂, α₃)    — 5 parameters */

/* basis_function of approx (src/psd.jl:214) */
#define PIORAN_BASIS_SHO 0
#define PIORAN_BASIS_DRWCELERITE 1

typedef struct pioran_ctx pioran_ctx;

/* Parameters of  approx(psd_model, f_min, f_max, n_components, norm, S_low, S_high; is_integrated_power,
 * basis_function)  (src/psd.jl:214) that do not vary inside a batch. */
typedef struct pioran_approx_spec {
    int32_t psd_model;           /* PIORAN_PSD_*                                  */
    int32_t n_components;        /* J                                             */
    int32_t basis;               /* PIORAN_BASIS_*                                */
    int32_t is_integrated_power; /* 1 (reference default) or 0                    */
    double f_min, f_max;         /* frequency range of the time series            */
    double S_low, S_high;        /* reference defaults 20, 20                     */
} pioran_approx_spec;

const char *pioran_last_error(void);
/* Library/ABI version: major*10000 + minor*100 + patch. */
int pioran_version(void);

/* One column of a prior transform (quantile(d, u) of Distributions.jl, which the reference's samplers call:
 * examples/ultranest/single_pl.jl:96-104, docs/src/ultranest.md:165-190). */
#define PIORAN_PRIOR_UNIFORM 0      /* Uniform(p0, p1)                                                   */
#define PIORAN_PRIOR_UNIFORM_FROM 1 /* Uniform(theta[ref_col], p1): lower edge = an EARLIER column        */
#define PIORAN_PRIOR_LOGUNIFORM 2   /* LogUniform(p0, p1)                                                */
#define PIORAN_PRIOR_NORMAL 3       /* Normal(mean p0, standard deviation p1)                            */
#define PIORAN_PRIOR_LOGNORMAL 4    /* LogNormal(p0, p1)                                                 */
#define PIORAN_PRIOR_GAMMA 5        /* Gamma(shape p0 (integer, 1 ... 32), scale p1)                     */
typedef struct pioran_prior_spec {
    int32_t kind;                /* PIORAN_PRIOR_*                                                        */
    int32_t ref_col;             /* UNIFORM_FROM only                                                     */
    double p0, p1;
} pioran_prior_spec;

/* ---- context & resident time series -------------------------------------------------------------------- */
/* Binds a context to CUDA device `device` (must be compute capability 10.x).  Creates one stream. */
int pioran_ctx_create(int device, pioran_ctx **out);
int pioran_ctx_destroy(pioran_ctx *ctx);
/* One context over several devices of the box, for a caller that is ONE process with one likelihood callback (the
 * reference's samplers: examples/ultranest/single_pl.jl:113-117; dispatch of src/scalable_GP.jl:24-40, 162-166).
 * pioran_series_upload places the series on every device; the batched host-pointer entries (pioran_approx_logl,
 * pioran_approx_logl_logshift, pioran_approx_logl_sine(_grad), pioran_approx_logl_grad, pioran_celerite_logl, pioran_direct_logl) cut their B parameter vectors into ndev
 * contiguous slices, run each slice on its device concurrently and write the results straight into the caller's arrays -
 * the slices are independent, so no collective is involved.  Every other entry runs on devices[0]; the device-pointer
 * entries (_dev) and pioran_ctx_set_stream need a single-device context and return PIORAN_EUNSUPPORTED on a group. */
int pioran_ctx_create_multi(const int *devices, int ndev, pioran_ctx **out);
/* Number of devices behind a context (1 for pioran_ctx_create). */
int pioran_ctx_device_count(pioran_ctx *ctx);
/* Use an external stream (e.g. torch's current stream, passed as its cudaStream_t cast to void*) for all
 * subsequent launches of this context; NULL restores the context's own stream. */
int pioran_ctx_set_stream(pioran_ctx *ctx, void *cuda_stream);
int pioran_ctx_synchronize(pioran_ctx *ctx);
/* Number of CUDA kernels this context has launched since creation (bench.py's gpu_launches). */
int64_t pioran_ctx_launch_count(pioran_ctx *ctx);
/* Device time (ms, CUDA events on the context's stream) of the most recent main-kernel launch — the batched
 * celerite kernel K2, the scan K3 or the dense K4.  Waits for that launch to finish. */
int pioran_ctx_last_kernel_ms(pioran_ctx *ctx, double *ms);
/* Name of the kernel that launch ran, with its template integers, as a NUL-terminated string in buf[len]: one format per
 * family, e.g. "blocked<5,5,true,16>", "blocked_wide<9,10,4>", "shared<8,4>", "shared_pair<4,8>", "generic<5,12>",
 * "wide_reg<7>", "wide", "blocked_grad<3,3,false,4>", "grad<4,8>", "grad_pipe<8,5>", "wide_grad<5>", "jvp<4>",
 * "scan_finish", "dense_finish".  Empty before the first launch.  Which kernel serves a shape is an implementation
 * detail that may change between versions; this is for tests and profiles.  PIORAN_EINVAL when len is too small for the
 * name; PIORAN_EUNSUPPORTED on a device group. */
int pioran_ctx_last_kernel_name(pioran_ctx *ctx, char *buf, int len);

/* Uploads one time series (τ, y, σ²) — the (x, Y, diag Σy) of logpdf(f(t, σ²), y), src/scalable_GP.jl:162-166 —
 * and keeps it resident.  t must be strictly increasing.  A sampler uploads once and evaluates ~1e5 times. */
int pioran_series_upload(pioran_ctx *ctx, int64_t N, const double *t, const double *y, const double *s2,
                         int *series_id);
int pioran_series_free(pioran_ctx *ctx, int series_id);
int pioran_series_length(pioran_ctx *ctx, int series_id, int64_t *N);

/* ---- K1: approx (src/psd.jl:214-289) --------------------------------------------------------------------- */
/* theta: [B × (n_psd_par + 1)] row-major = psd parameters…, norm.  Outputs a,b,c,d: [B × Jt] row-major with
 * Jt = J (SHO) or 2J (DRWCelerite: J celerite terms followed by J DRW terms, src/psd.jl:264-275). */
int pioran_approx_coeffs(pioran_ctx *ctx, const pioran_approx_spec *spec, int B, const double *theta,
                         double *a, double *b, double *c, double *d);

/* approx() of a continuum plus narrow PSD features (src/psd.jl:15-44 convert_feature / get_covariance_from_psd, :221-243,
 * :254-259, :277-282; test/test_psd.jl:206-285): each QPO(S0, f0, Q) becomes one more celerite term
 * (a, b, c, d) = (S0 w0 Q/4, a/D, w0/(2Q), c D), D = sqrt(4 Q^2 - 1), w0 = 2 pi f0, divided by the continuum's PSD at the first
 * grid point, normalised together with the continuum (its integral joins the norm when is_integrated_power = 1) and doubled.
 * theta: [B x (n_psd_par + 1 + 3 n_features)] = psd parameters..., norm, then (S0, f0, Q) per feature.  Outputs: [B x (Jt +
 * n_features)], the Jt continuum terms of pioran_approx_coeffs followed by the feature terms.  1 <= n_features <= 8. */
int pioran_approx_coeffs_features(pioran_ctx *ctx, const pioran_approx_spec *spec, int n_features, int B,
                                  const double *theta, double *a, double *b, double *c, double *d);

/* ---- K2: celerite log-likelihood ------------------------------------------------------------------------ */
/* Drop-in for  logl(a, b, c, d, τ, y, σ2)  (src/celerite_solver.jl:312-334) over a batch of B coefficient sets,
 * [B × Jt] row-major each.  mu/nu: per-set constant mean and variance scale (y−μ, ν·σ²; NULL → 0 / 1), the two
 * θ-dependent scalars of the samplers' likelihoods (examples/ultranest/single_pl.jl:70-73).
 * y_batch: NULL, or [B × N] per-set data vectors replacing the resident y (custom mean functions, log-shift
 * transforms); s2_batch likewise for σ².  logl_out: [B]. */
int pioran_celerite_logl(pioran_ctx *ctx, int series_id, int B, int Jt,
                         const double *a, const double *b, const double *c, const double *d,
                         const double *mu, const double *nu,
                         const double *y_batch, const double *s2_batch, double *logl_out);

/* Fused  approx(...) + logpdf(ScalableGP(μ, 𝓡)(t, ν·σ²), y)  for B parameter vectors on each of S resident series.
 * specs: [S] (f_min/f_max differ per series; J, basis, model must agree).  theta: [B × (n_psd_par+3)] row-major =
 * psd parameters…, norm, ν, μ — shared by all series when theta_per_series == 0, else [S × B × (n_psd_par+3)].
 * y_batch: NULL or [S × B × Nmax]-free form is not supported here (use pioran_celerite_logl).  logl_out: [S × B]. */
int pioran_approx_logl(pioran_ctx *ctx, int S, const int *series_ids, const pioran_approx_spec *specs,
                       int B, const double *theta, int theta_per_series, double *logl_out);

/* approx(continuum + QPO features) + logpdf for B parameter vectors on one resident series: theta [B x (n_psd_par + 3 +
 * 3 n_features)] = psd parameters..., norm, nu, mu, then (S0, f0, Q) per feature.  The feature terms' decay rates and frequencies
 * depend on theta, so the sweep is the explicit-coefficient kernel of pioran_celerite_logl (ranks up to 160). */
int pioran_approx_features_logl(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int n_features, int B,
                                const double *theta, double *logl_out);

/* Fused path for log-normally distributed series (reference: docs/src/timeseries.md:16-21 and the likelihood of
 * docs/src/ultranest.md:197-217):  yn = log(y - c),  sigma2 = nu * sigma^2 / (y - c)^2,  logpdf(ScalableGP(mu, R)(t, sigma2), yn).
 * theta: [B x (n_psd_par+4)] row-major = psd parameters..., norm, nu, mu, c.  The transform runs on the device (one pass
 * over B x N, in theta-chunks of at most 1 GiB) in front of the same K1 + K2 as pioran_approx_logl; y - c <= 0 gives a
 * NaN log-likelihood (the reference throws DomainError).  One resident series, ranks <= 64.  logl_out: [B]. */
int pioran_approx_logl_logshift(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int B,
                                const double *theta, double *logl_out);

/* Same as pioran_approx_logl with θ and the result resident in device memory; asynchronous on the context's
 * stream (no host synchronisation).  theta_dev: [S or 1][B][n_psd_par+3]; logl_dev: [S × B]. */
int pioran_approx_logl_dev(pioran_ctx *ctx, int S, const int *series_ids, const pioran_approx_spec *specs,
                           int B, const double *theta_dev, int theta_per_series, double *logl_dev);

/* ---- K5: gradient of the fused path (widening row, SURVEY 8f #1) -------------------------------------------
 * Replaces  ForwardDiff.gradient(θ -> logpdf(ScalableGP(μ, approx(𝓟(θ…), f_min, f_max, J, norm))(t, ν·σ²), y), θ)
 * (reference test/test_likelihood.jl:24-43,55; the NUTS runs of examples/turing_distributed/single_pl.jl): forward-mode
 * derivatives pushed through the same two kernels, one warp per (parameter vector, PSD parameter or ν); the μ and norm
 * partials come from the same sweeps (right-hand-side tangent; homogeneity of K in (norm, ν)).
 * theta: [B × (n_psd_par+3)] = psd parameters…, norm, ν, μ.  logl_out: [B] or NULL.  grad_out: [B × (n_psd_par+3)],
 * ∂logℒ/∂θ in the column order of theta. */
int pioran_approx_logl_grad(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int B,
                            const double *theta, double *logl_out, double *grad_out);
/* Same with θ and the results resident in device memory (asynchronous on the context's stream once the work-item list is
 * uploaded). */
int pioran_approx_logl_grad_dev(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int B,
                                const double *theta_dev, double *logl_dev, double *grad_dev);

/* Which kernel sweeps the fused (approx) path at ranks <= 63.  PIORAN_SWEEP_AUTO (default): the tensor-pipe kernel
 * (csrc/blocked.cuh: the recursion of src/celerite_solver.jl:69-98 blocked over 8 steps, its O(R^2) work on FP64 mma.sync);
 * PIORAN_SWEEP_SCALAR: the scalar-pipe kernel (csrc/celerite.cuh), kept for ranks 64, explicit coefficients and as the
 * in-process cross-check of the blocked one.  Both evaluate the same log-likelihood. */
#define PIORAN_SWEEP_AUTO 0
#define PIORAN_SWEEP_SCALAR 1
int pioran_ctx_set_sweep_kernel(pioran_ctx *ctx, int which);

/* Gradient of the log-normal likelihood of pioran_approx_logl_logshift: theta [B x (n_psd_par+4)] = psd parameters..., norm, nu, mu, c;
 * grad_out [B x (n_psd_par+4)] in the column order of theta, d/dc included (the reference differentiates this model with
 * ForwardDiff like any other: docs/src/ultranest.md:197-217, test/test_likelihood.jl:55).  The shift moves the data:
 * d yn/dc = -1/(y - c), d sigma2/dc = 2 nu sigma^2/(y - c)^3, carried as one more tangent direction of the blocked gradient kernel.
 * SingleBendingPowerLaw, ranks <= 62.  logl_out: [B] or NULL. */
int pioran_approx_logl_logshift_grad(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int B,
                                     const double *theta, double *logl_out, double *grad_out);

/* Sinusoidal mean (examples/ultranest/single_pl_periodicity.jl, the reference's periodicity search):
 *   logl = logpdf(ScalableGP(m, approx(P, f_min, f_max, J, norm))(t, nu*sigma^2), y),   m(t) = mu + A*sin(2*pi*t/T0 + phi)
 * theta: [B x (n_psd_par+6)] row-major = psd parameters..., norm, nu, mu, A, phi, T0.  y - A*sin(...) is formed on the device
 * (one pass over B x N, in theta-chunks of at most 1 GiB) in front of the same K1 + K2 as pioran_approx_logl; mu stays the
 * sweep's scalar, so A = 0 gives pioran_approx_logl's value bit for bit.  Non-finite results are returned as data.  One
 * resident series, ranks <= 64 (PIORAN_EUNSUPPORTED above).  logl_out: [B]. */
int pioran_approx_logl_sine(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int B,
                            const double *theta, double *logl_out);
/* Gradient of pioran_approx_logl_sine: grad_out [B x (n_psd_par+6)] in the column order of theta.  The partials of A, phi and
 * T0 are the innovations of three data rows whose right-hand sides are d(y - m)/d(A, phi, T0), carried by one more warp of the
 * blocked gradient kernel.  Single- and DoubleBendingPowerLaw, ranks <= 62 (PIORAN_EUNSUPPORTED above, and under
 * PIORAN_SWEEP_SCALAR).  logl_out: [B] or NULL. */
int pioran_approx_logl_sine_grad(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int B,
                                 const double *theta, double *logl_out, double *grad_out);

/* ---- K5g: forward-mode derivatives of the explicit-coefficient likelihood ----------------------------------
 * d/dε of pioran_celerite_logl along P directions per parameter vector (ForwardDiff's chunk over logl): for set i and
 * direction p,  logl(a_i + ε da_ip, b_i + ε db_ip, c_i + ε dc_ip, d_i + ε dd_ip, τ, ỹ, σ̃²)  with  ỹ = y_i + ε dy_ip − (μ_i + ε dμ_ip)
 * and  σ̃² = (ν_i + ε dν_ip)(s2_i + ε ds2_ip);  y_i, s2_i are the resident series or the rows of y_batch/s2_batch.
 * Tangent arrays may be NULL (zero): da/db/dc/dd [B × P × Jt], dmu/dnu [B × P], dy/ds2 [B × P × N].  logl_out [B] or NULL;
 * dlogl_out [B × P].  A term that is real for every set of the batch (b = d = 0) ignores its db, dd (exact: ∂k/∂b and ∂k/∂d
 * vanish there).  Ranks <= 96 (PIORAN_EUNSUPPORTED above); P < 1, a NULL dlogl_out, an unknown series or B·P beyond
 * INT_MAX give PIORAN_EINVAL.  Data tangents are uploaded in θ-chunks of at most 1 GiB. */
int pioran_celerite_logl_jvp(pioran_ctx *ctx, int series_id, int B, int Jt, int P,
                             const double *a, const double *b, const double *c, const double *d,
                             const double *mu, const double *nu, const double *y_batch, const double *s2_batch,
                             const double *da, const double *db, const double *dc, const double *dd,
                             const double *dmu, const double *dnu, const double *dy, const double *ds2,
                             double *logl_out, double *dlogl_out);
/* Gradient of pioran_approx_features_logl: theta and grad_out [B × (n_psd_par + 3 + 3 n_features)], same column order
 * (psd parameters…, norm, ν, μ, (S₀, f₀, Q)…).  The coefficients and their tangents along every θ column are formed on the
 * device (K1 on dual numbers with the feature branch) and swept by the K5g kernel.  logl_out [B] or NULL.  Ranks <= 96,
 * 1 … 8 features (PIORAN_EUNSUPPORTED beyond 8). */
int pioran_approx_features_logl_grad(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int n_features, int B,
                                     const double *theta, double *logl_out, double *grad_out);

/* ---- K5r: reverse-mode gradient of the explicit-coefficient likelihood -------------------------------------
 * For every set i of pioran_celerite_logl's inputs (same arguments), one backward sweep gives logL_i and its gradient with
 * respect to a, b, c, d (ga … gd [B × Jt]), μ_i and ν_i (gmu, gnu [B]) and the data row as it enters, ỹ = y − μ and σ̃² = ν·s2
 * (gy, gs2 [B × N]; y, s2 are the resident series or the rows of y_batch/s2_batch).  It is the function K5g differentiates:
 * <gradient, v> = pioran_celerite_logl_jvp along v.  A term real for every set of the batch (b = d = 0) gets gb = gd = 0 exactly.
 * Every output may be NULL, but at least one gradient output must be given.  Ranks <= 96 (PIORAN_EUNSUPPORTED above); no
 * gradient output, an unknown series or B < 1 give PIORAN_EINVAL.  The workspace (per-step values and checkpoints of the state,
 * about (2R + 2)·N + (⌈N/K⌉ + K)·256·⌈R/16⌉² doubles per set with K ≈ √N) is bounded by processing the batch in θ-chunks of at
 * most 1 GiB (pioran_ctx_set_vjp_workspace). */
int pioran_celerite_logl_vjp(pioran_ctx *ctx, int series_id, int B, int Jt,
                             const double *a, const double *b, const double *c, const double *d,
                             const double *mu, const double *nu, const double *y_batch, const double *s2_batch,
                             double *logl_out, double *ga, double *gb, double *gc, double *gd,
                             double *gmu, double *gnu, double *gy, double *gs2);
/* Same arguments, columns and limits as pioran_approx_features_logl_grad, computed by one K5r sweep and a contraction with the
 * coefficient tangents instead of one forward direction per θ column. */
int pioran_approx_features_logl_grad_reverse(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int n_features,
                                             int B, const double *theta, double *logl_out, double *grad_out);
/* Cap in bytes of the K5r workspace of one θ-chunk (0 = 1 GiB, the default).  The result does not depend on it; a small cap
 * splits a batch into many chunks (one set per chunk at least). */
int pioran_ctx_set_vjp_workspace(pioran_ctx *ctx, long long bytes);

/* ---- K3: long single series, parallel-in-time (same recursion, N ~ 1e6) --------------------------------- */
/* Prior transform on the device (the `prior_transform(cube)` callback of examples/ultranest/single_pl.jl:96-104, batched):
 * cube [B x ncol] unit-cube points -> theta_out [B x ncol], columns left to right.  pioran_prior_transform_logl does the
 * transform and the fused likelihood of pioran_approx_logl (one series) in one call - the parameter vectors never leave the
 * device unless theta_out is given (ncol must be n_psd_par + 3: psd parameters, norm, nu, mu). */
int pioran_prior_transform(pioran_ctx *ctx, int ncol, const pioran_prior_spec *priors, int B, const double *cube,
                           double *theta_out);
int pioran_prior_transform_logl(pioran_ctx *ctx, int series_id, const pioran_approx_spec *spec, int ncol,
                                const pioran_prior_spec *priors, int B, const double *cube, double *theta_out,
                                double *logl_out);

/* Same value as pioran_celerite_logl with B small, computed by the chunked associative-scan formulation. */
/* pioran_celerite_logl and pioran_approx_logl hand calls with at most 4 parameter vectors on a long series (fused path: at
 * least 4 096 steps, 2 048 at rank <= 32; explicit coefficients: half of that; rank <= 64, no per-vector data) to the
 * parallel-in-time path: a lone sequential sweep costs 0.5-1.5 us per step whatever the batch.  enabled = 0 keeps them on the
 * sequential kernels (default: enabled). */
int pioran_ctx_set_auto_scan(pioran_ctx *ctx, int enabled);

/* Self-check and Newton refinement of the parallel-in-time path.  Its composites lose accuracy where the covariance is
 * ill-conditioned (steep PSD slopes), so every call verifies itself: at each chunk boundary the 8 steps after it are
 * swept twice - continuing the sweep of the previous chunk, and from the state the scan computed - and the difference
 * of their contributions to log L, scaled to the chunk length and summed over the boundaries, estimates the deviation
 * from the sequential sweep.  Parameter vectors whose estimate exceeds tol * max(1, |log L|) get their chunk states
 * corrected by Newton steps whose residual is the exact recursion itself (the last pass of the path is run chunk by
 * chunk and returns the state every chunk leaves behind; the corrections follow a linear recurrence along the chunks),
 * each verified the same way.  A parameter vector is accepted when its estimate meets tol, or when at least two Newton
 * steps were taken, the estimate stalls (within 4x of the previous one, below 1000 x cap) and the value itself moved
 * by no more than cap * max(1, |log L|) between the last two steps: what is left then is the rounding noise of an FP64
 * evaluation of that covariance - any two FP64 routes differ by it, the sequential sweep's distance from an 80-bit
 * evaluation included.  What still fails (composites breaking down on a barely
 * positive definite covariance) is evaluated by the sequential kernel (reference: src/celerite_solver.jl:312-334 has
 * one formulation only).  Defaults: tol = 1e-10, floor cap = 1e-7; tol <= 0 disables refinement and fallback (the
 * estimate is still computed); cap <= 0 never accepts a stalled iteration.  pioran_ctx_last_scan_check reports the
 * largest relative estimate among the results of the last call, how many parameter vectors went to the sequential
 * kernel and how many were accepted after a refinement pass (any pointer may be NULL); after
 * pioran_celerite_scan_range_end it reports that range's part of the estimate in log L units (no refinement across
 * ranks: the caller decides).  pioran_ctx_last_scan_history returns, for parameter vector `index` of the last call,
 * the relative estimate and the value after every pass it went through (pass 0: the scan's states; pass 1: the same
 * states swept chunk by chunk; pass k >= 2: after k - 1 Newton steps); *n_passes = how many there were. */
int pioran_ctx_set_scan_tolerance(pioran_ctx *ctx, double tol);
int pioran_ctx_last_scan_check(pioran_ctx *ctx, double *estimate, int *n_fallback, int *n_refined);
int pioran_ctx_set_scan_floor_cap(pioran_ctx *ctx, double cap);
int pioran_ctx_last_scan_history(pioran_ctx *ctx, int index, int max_passes, double *estimates, double *values,
                                 int *n_passes);

/* Number of time-axis chunks per parameter vector used by pioran_celerite_logl_scan (0 = automatic: two per SM, at
 * least 64 steps each).  The result does not depend on it beyond rounding; tests use it to exercise the scan on short
 * series. */
int pioran_ctx_set_scan_chunks(pioran_ctx *ctx, int chunks);
int pioran_celerite_logl_scan(pioran_ctx *ctx, int series_id, int B, int Jt,
                              const double *a, const double *b, const double *c, const double *d,
                              const double *mu, const double *nu, double *logl_out);

/* The same path with the TIME AXIS split across GPUs (SURVEY 8e): every rank holds the series, folds its own step range
 * [n_lo, n_hi) and returns the range's composite scan element (pioran_scan_composite_doubles() doubles, ~97 KB);
 * the ranks all-gather those (NCCL / MPI — outside this library); each rank then passes the composites of the ranges that
 * precede its own, in time order, and gets (sum log|D_n|, sum z_n^2/D_n) over its range; the caller all-reduces the two
 * sums and forms  logL = -sums[0]/2 - sums[1]/2 - N log(2 pi)/2  (src/celerite_solver.jl:333).  One coefficient set per
 * call.  max_prev = upper bound of nprev (workspace sizing).  begin/end must be called in pairs on the same context. */
int pioran_scan_composite_doubles(void);
int pioran_celerite_scan_range_begin(pioran_ctx *ctx, int series_id, int Jt,
                                     const double *a, const double *b, const double *c, const double *d,
                                     const double *mu, const double *nu, int64_t n_lo, int64_t n_hi, int max_prev,
                                     double *composite_out);
int pioran_celerite_scan_range_end(pioran_ctx *ctx, int nprev, const double *composites_prev, double *sums_out);

/* Self-check data of the range pioran_celerite_scan_range_end just finished, out8 =
 *   [0]    this range's inner estimate (log L units; see pioran_ctx_set_scan_tolerance),
 *   [1..2] (sum log|D|, sum z^2/D) of the first out8[5] steps of the range, swept from the state the earlier composites gave,
 *   [3..4] the same sums over the out8[6] steps AFTER the range, swept on from this range's own final state,
 *   [5], [6] those step counts (0 at the two ends of the series; [6] is also 0 after a range of odd length - split
 *            the time axis at even steps),  [7] the scale (sub-chunk length / check length).
 * The hand-over from rank r-1 to rank r is consistent when [3..4] of r-1 equal [1..2] of r; the caller gathers the eight
 * values of every rank, adds scale * (|d sum log|D|| + |d sum z^2/D|) / 2 of each hand-over to the inner estimates and
 * falls back to a sequential evaluation when the total exceeds its tolerance (pioran.jl_b200/parallel.py:
 * scan_logl_sharded does exactly that). */
int pioran_celerite_scan_range_check(pioran_ctx *ctx, double *out8);

/* ---- K4: dense cross-check ------------------------------------------------------------------------------- */
/* Drop-in for  log_likelihood_direct(cov, t, y, σ²)  (src/direct_solver.jl:6-21) with the kernel of
 * src/Celerite.jl:42-44 summed over terms.  Returns +NLL like the reference (tests negate it,
 * test/test_likelihood.jl:54).  info_out[i] = 0, or k>0 when the leading minor of order k is not positive
 * definite (the reference throws PosDefException; here nll_out[i] = NaN). */
int pioran_direct_logl(pioran_ctx *ctx, int series_id, int B, int Jt,
                       const double *a, const double *b, const double *c, const double *d,
                       const double *mu, const double *nu, double *nll_out, int *info_out);

/* ---- widening rows (SURVEY 8f #2, #3): posterior mean and GP draws ------------------------------------------ */
/* Batched drop-in for  predict(cov, τ, t, y, σ²) = pred(a, b, c, d, τ, t, y, σ²)  (src/celerite_solver.jl:348-483), the
 * routine behind  mean(posterior(f(t, σ²), y), τ)  (src/scalable_GP.jl:61-67, 84-85): for each of the B coefficient sets
 * the posterior mean  mu_i + K(τ, t) (K(t, t) + diag(nu_i σ²))⁻¹ (y − mu_i)  at the M ascending points tau.
 * mean_out is [B × M] row-major; mu/nu as in pioran_celerite_logl (NULL → 0 / 1). */
int pioran_celerite_predict(pioran_ctx *ctx, int series_id, int B, int Jt,
                            const double *a, const double *b, const double *c, const double *d,
                            const double *mu, const double *nu, int64_t M, const double *tau, double *mean_out);
/* Batched drop-in for  simulate(rng, cov, t, σ²) = sim(rng, a, b, c, d, t, σ²)  (src/celerite_solver.jl:497-549), behind
 * rand(f(t, σ²))  (src/scalable_GP.jl:133-155): y_i = L_i q_i with L_i the celerite factor of K_i + diag(nu_i σ²) on the
 * series' times.  The standard-normal draws q [B × N] are the caller's (Julia's randn stream cannot be reproduced on
 * the device); y_out is [B × N].  A non-positive pivot gives NaN from that step on (the reference raises DomainError). */
int pioran_celerite_simulate(pioran_ctx *ctx, int series_id, int B, int Jt,
                             const double *a, const double *b, const double *c, const double *d,
                             const double *nu, const double *q, double *y_out);
/* Posterior predictive variance (K6): for each of the B coefficient sets the variance of the latent f at the M ascending
 * points tau,  var_out[i][m] = k_i(0) − k_i(τ_m, t)ᵀ (K_i(t, t) + diag(nu_i σ²))⁻¹ k_i(τ_m, t)  — the diagonal of
 * predict_cov (src/direct_solver.jl:28-119) behind var / std of a PosteriorGP, without measurement noise and independent of
 * mu.  O((N + M)·R²) per set from the factor of pioran_celerite_predict; ranks up to 128 (PIORAN_EUNSUPPORTED above).
 * mean_out [B × M] (or NULL) is what pioran_celerite_predict returns for the same arguments, bit for bit.  A set whose
 * factor has a pivot D_n <= 0 gets NaN in every entry of its var_out row.  Arguments are checked as in
 * pioran_celerite_predict; on a device group the call runs on the first device. */
int pioran_celerite_predict_var(pioran_ctx *ctx, int series_id, int B, int Jt,
                                const double *a, const double *b, const double *c, const double *d,
                                const double *mu, const double *nu, int64_t M, const double *tau,
                                double *mean_out, double *var_out);
/* Posterior draws (K7): for each of the B coefficient sets, S draws of  rand(fp(τ, sigma2_tau))  for the posterior
 * fp = posterior(f(t, nu_i σ²), ỹ_i) — the latent f at the M ascending points tau conditioned on the data, plus independent
 * noise of variance sigma2_tau (AbstractGPs' σ² of fp(τ, σ²); 1e-18 is its default).  ỹ_i is the resident y, or row i of
 * y_batch [B × N] when given.  Matheron's rule on the merged grid G of t and τ (a data point first at a tie): a prior draw
 * u = L^G √D^G q on G, then draw = mu_i + u(τ) + K(τ, t) K̃⁻¹ (ỹ − mu_i − u(t)).  q [B × S × (N + M)] holds standard normals
 * in merged-grid order (the caller's, as for pioran_celerite_simulate); draws_out is [B × S × M].  For the same q this is
 * not the draw a dense Cholesky of the posterior covariance gives; its distribution is the same.  O((N + M)·R²) per set
 * for the two factors, O((N + M)·R) per draw; ranks up to 128 (PIORAN_EUNSUPPORTED above).  PIORAN_EINVAL for NULL
 * pointers, B, Jt, M or S < 1, descending tau, sigma2_tau < 0 or NaN, and repeated tau with sigma2_tau == 0 (the merged
 * covariance is then singular).  A set with a pivot <= 0 in either factor gets NaN in all of its S·M draws.  A device
 * group splits the sets over its devices. */
int pioran_celerite_posterior_draws(pioran_ctx *ctx, int series_id, int B, int Jt,
                                    const double *a, const double *b, const double *c, const double *d,
                                    const double *mu, const double *nu, const double *y_batch,
                                    int64_t M, const double *tau, double sigma2_tau,
                                    int S, const double *q, double *draws_out);
/* Posterior covariance (K8): for each of the B coefficient sets the full covariance of the latent f at the M ascending points
 * tau,  cov_out[i][m][m'] = k_i(τ_m, τ_m') − k_i(τ_m, t)ᵀ (K_i(t, t) + diag(nu_i σ²))⁻¹ k_i(t, τ_m')  — predict_cov
 * (src/direct_solver.jl:28-119) behind cov / mean_and_cov of a PosteriorGP, without measurement noise and independent of mu.
 * cov_out is [B × M × M] row-major and exactly symmetric; its diagonal is pioran_celerite_predict_var's variance up to
 * rounding.  O((N + M)·R² + M·(N + M)·R) per set from the factor of pioran_celerite_predict: K6 adds two vectors per point,
 * then one walk per column over the merged grid of t and τ.  mean_out [B × M] (or NULL) is what pioran_celerite_predict
 * returns for the same arguments, bit for bit.  Ranks up to 128 (PIORAN_EUNSUPPORTED above); arguments are checked as in
 * pioran_celerite_predict_var.  A set whose factor has a pivot D_n <= 0 gets NaN in its whole matrix.  The device workspace
 * and output of one step is at most 1 GiB (pioran_ctx_set_postcov_workspace): the sets are processed in θ-chunks, and a set
 * whose matrix alone exceeds the cap in column ranges.  A device group splits the sets over its devices. */
int pioran_celerite_predict_cov(pioran_ctx *ctx, int series_id, int B, int Jt,
                                const double *a, const double *b, const double *c, const double *d,
                                const double *mu, const double *nu, int64_t M, const double *tau,
                                double *mean_out, double *cov_out);
/* Cap in bytes of the device workspace plus output of one step of pioran_celerite_predict_cov (0 = 1 GiB, the default).
 * The result does not depend on it; a small cap splits a batch into many θ-chunks, and a set into column ranges. */
int pioran_ctx_set_postcov_workspace(pioran_ctx *ctx, long long bytes);
/* Generalised Lomb–Scargle periodograms (K9) of B series on the times of one resident series: the floating-mean periodogram
 * (Zechmeister & Kürster 2009) with the :standard normalisation, which LombScargle.jl computes by default (fit_mean,
 * center_data) and the posterior predictive checks of src/plots_diagnostics.jl:532-546 take for one simulated series per
 * posterior sample.  y_batch [B × N] (NULL: the resident y, B must be 1); weighted = 1: weights 1/s2 of the resident series
 * (LombScargle.jl's `errors`), 0: equal weights.  freq [F] > 0 and finite, any order, in the inverse unit of t.  power_out
 * [B × F] row-major, in [0, 1].  Where the formula divides zero by zero (an all-zero row, N = 1, a frequency at which the
 * basis is degenerate on these times) the value is NaN; that is data, not an error.  PIORAN_EINVAL for NULL ctx, freq or
 * power_out, B or F < 1, a NULL y_batch with B > 1, a frequency that is not positive and finite, an unknown series, and
 * weighted with an s2 of the series that is not positive and finite.  Each value is summed in the same order whatever B,
 * the chunking or the row's position, so a row's periodogram is the same bit for bit in any batch.  A device group splits
 * the rows over its devices. */
int pioran_lombscargle(pioran_ctx *ctx, int series_id, int B, const double *y_batch, int weighted,
                       int64_t F, const double *freq, double *power_out);
/* Cap in bytes of the device workspace plus output of one step of pioran_lombscargle (0 = 1 GiB, the default).  The result
 * does not depend on it; a small cap splits the frequencies and the rows into many chunks. */
int pioran_ctx_set_lsp_workspace(pioran_ctx *ctx, long long bytes);

#ifdef __cplusplus
}
#endif
#endif /* PIORAN_B200_H */
