/*
 * oracle_sine.c — forward-mode restatement of the likelihood with a sinusoidal mean, the reference's periodicity run
 * (examples/ultranest/single_pl_periodicity.jl).  TEST INFRASTRUCTURE ONLY: the reference of pioran_approx_logl_sine_grad in
 * tests/test_gpu_sine.py.
 *
 * It is the dual-number sweep of oracle/pioran_oracle_grad.c (included below, unchanged: approx on duals, then the reference's
 * celerite recursion on duals) with the data row y − m(t), m(t) = μ + A·sin(2π·t/T₀ + ϕ), carrying the tangents of μ, A, ϕ and
 * T₀.  Compiled with the oracle's flags (oracle/Makefile: no contraction of a*b+c) together with oracle/pioran_oracle.c;
 * oracle_sine_ld.c compiles the same source in x87 80-bit arithmetic for conditioning triage.
 */
#include "pioran_oracle_grad.c"

#ifdef ORC_GRAD_LONG_DOUBLE
#define ORC_SINE_ENTRY orc_approx_logl_sine_grad_batch_ld
#else
#define ORC_SINE_ENTRY orc_approx_logl_sine_grad_batch
#endif

static inline dual dsin(dual a) { return dmk(RM(sin)(a.v), RM(cos)(a.v) * a.d); }

/* θ row = [psd params…, norm, ν, μ, A, ϕ, T₀]; logl_out [B] (may be NULL), grad_out [B × (n_psd_par + 6)] = ∂logL/∂θ, one
 * forward sweep per direction. */
void ORC_SINE_ENTRY(int model, int n_psd_par, int B, const double *theta, double f_min, double f_max, int J, double S_low,
                    double S_high, int is_integrated_power, int basis, int64_t N, const double *t, const double *y,
                    const double *s2_base, double *logl_out, double *grad_out, int nthreads)
{
    const int P = n_psd_par + 6;
#ifdef _OPENMP
    if (nthreads < 1) nthreads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 1) num_threads(nthreads) collapse(2)
#endif
    for (int i = 0; i < B; i++) {
        for (int k = 0; k < P; k++) {
            const double *th = theta + (size_t)i * P;
            dual par[11];
            for (int q = 0; q < P; q++) par[q] = dmk(th[q], q == k ? 1.0 : 0.0);
            dual norm = par[n_psd_par], nu = par[n_psd_par + 1], mu = par[n_psd_par + 2];
            dual A = par[n_psd_par + 3], phi = par[n_psd_par + 4], T0 = par[n_psd_par + 5];
            int Jt_max = 2 * J;
            dual *ab = (dual *)malloc(sizeof(dual) * 2 * Jt_max);
            real *cd = (real *)malloc(sizeof(real) * 2 * Jt_max);
            dual *yy = (dual *)malloc(sizeof(dual) * N);
            dual *ss = (dual *)malloc(sizeof(dual) * N);
            for (int64_t n = 0; n < N; n++) {
                dual arg = dadd(ddiv(dk(2 * R_PI * (real)t[n]), T0), phi);          /* 2π·t/T₀ + ϕ */
                yy[n] = dsub(dk(y[n]), dadd(mu, dmul(A, dsin(arg))));              /* y − (μ + A·sin) */
                ss[n] = dmulc(nu, s2_base[n]);
            }
            int Jt = approx_dual(model, par, f_min, f_max, J, norm, S_low, S_high, is_integrated_power, basis, ab,
                                 ab + Jt_max, cd, cd + Jt_max);
            dual r = dmk(NAN, NAN);
            if (Jt > 0) r = celerite_logl_dual(Jt, ab, ab + Jt_max, cd, cd + Jt_max, N, t, yy, ss);
            if (logl_out && k == 0) logl_out[i] = (double)r.v;
            grad_out[(size_t)i * P + k] = (double)r.d;
            free(ab); free(cd); free(yy); free(ss);
        }
    }
}
