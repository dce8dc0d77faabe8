/*
 * oracle_jvp.c — forward-mode restatement of the explicit-coefficient likelihood with tangents on EVERY input (a, b, c, d, μ, ν,
 * y, σ²), and of the likelihood with PSD features on dual numbers.  TEST INFRASTRUCTURE ONLY: the reference of the K5g kernel
 * (pioran.jl_b200/csrc/jvp.cuh) and of pioran_approx_features_logl_grad in tests/test_gpu_jvp.py.
 *
 * The sweep is the reference's own algorithm, not the kernel's: src/celerite_solver.jl:312-334 (init_semi_separable! with the
 * lower triangle S, then the forward and backward substitutions of solve_prec!), restated on duals exactly like
 * celerite_logl_dual of oracle/pioran_oracle_grad.c but with c and d carrying tangents too, so cos, sin and φ are computed on
 * duals.  Every term takes two rows (a real term is a complex one with b = d = 0), as in the oracle.  The value part performs the
 * operations of orc_celerite_logl (oracle/pioran_oracle.c) in the same order, so with zero tangents it is that oracle bit for bit.
 * The feature branch follows orc_approx_features (src/psd.jl:15-44, 214-289) on duals.
 *
 * One direction per sweep (a dual carries one partial); the batched entries loop over directions.  Compiled with the oracle's
 * flags (oracle/Makefile: no contraction of a*b+c) together with oracle/pioran_oracle.c, which provides the spectral grid and
 * matrix (orc_build_approx); oracle_jvp_ld.c compiles the same source in x87 80-bit arithmetic for conditioning triage.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

void orc_build_approx(int J, double f0, double fM, int basis, double *fj, double *B);

#ifdef ORC_JVP_LONG_DOUBLE
typedef long double real;
#define RM(f) f##l
#define R_PI 3.14159265358979323846264338327950288L
#define ORC_JVP_ENTRY orc_celerite_logl_jvp_batch_ld
#define ORC_FEAT_ENTRY orc_approx_features_logl_grad_batch_ld
#else
typedef double real;
#define RM(f) f
#define R_PI M_PI
#define ORC_JVP_ENTRY orc_celerite_logl_jvp_batch
#define ORC_FEAT_ENTRY orc_approx_features_logl_grad_batch
#endif

typedef struct { real v, d; } dual;

static inline dual dk(real v) { dual r = {v, 0.0}; return r; }
static inline dual dmk(real v, real d) { dual r = {v, d}; return r; }
static inline dual dadd(dual a, dual b) { return dmk(a.v + b.v, a.d + b.d); }
static inline dual dsub(dual a, dual b) { return dmk(a.v - b.v, a.d - b.d); }
static inline dual dneg(dual a) { return dmk(-a.v, -a.d); }
static inline dual dmul(dual a, dual b) { return dmk(a.v * b.v, a.d * b.v + a.v * b.d); }
static inline dual dmulc(dual a, real c) { return dmk(a.v * c, a.d * c); }
static inline dual ddivc(dual a, real c) { return dmk(a.v / c, a.d / c); }
static inline dual ddiv(dual a, dual b) { real q = a.v / b.v; return dmk(q, (a.d - q * b.d) / b.v); }
static inline dual dlog(dual a) { return dmk(RM(log)(a.v), a.d / a.v); }
static inline dual dlogabs(dual a) { return dmk(RM(log)(RM(fabs)(a.v)), a.d / a.v); }
static inline dual dsqrt(dual a) { real r = RM(sqrt)(a.v); return dmk(r, a.d / (2.0 * r)); }
static inline dual dcos(dual a) { return dmk(RM(cos)(a.v), -RM(sin)(a.v) * a.d); }
static inline dual dsin(dual a) { return dmk(RM(sin)(a.v), RM(cos)(a.v) * a.d); }
static inline dual dexp(dual a) { real e = RM(exp)(a.v); return dmk(e, e * a.d); }
static inline dual datan2(dual y, dual x) { return dmk(RM(atan2)(y.v, x.v), (x.v * y.d - y.v * x.d) / (x.v * x.v + y.v * y.v)); }
static inline dual dpow(dual x, dual e)
{
    real p = RM(pow)(x.v, e.v);
    return dmk(p, p * (e.d * RM(log)(x.v) + e.v * x.d / x.v));
}

/* src/celerite_solver.jl:312-334 on duals; every input but t carries a tangent.  y = y − μ and s2 = ν σ² as the caller forms them. */
static dual celerite_logl_jvp(int Jt, const dual *a, const dual *b, const dual *c, const dual *d, int64_t N,
                              const double *t, const dual *y, const dual *s2)
{
    const int R = 2 * Jt;
    dual *S = (dual *)calloc((size_t)R * R, sizeof(dual));
    dual *phi = (dual *)malloc(sizeof(dual) * (size_t)R * (N > 1 ? N - 1 : 1));
    dual *U = (dual *)malloc(sizeof(dual) * (size_t)R * N);
    dual *V = (dual *)malloc(sizeof(dual) * (size_t)R * N);
    dual *D = (dual *)malloc(sizeof(dual) * N);
    dual *z = (dual *)malloc(sizeof(dual) * N);
    dual *f = (dual *)calloc(R, sizeof(dual));
    dual *g = (dual *)calloc(R, sizeof(dual));
    dual result = dmk(NAN, NAN);
    if (!S || !phi || !U || !V || !D || !z || !f || !g) goto done;

    dual suma = dk(0.0);
    for (int j = 0; j < Jt; j++) suma = dadd(suma, a[j]);
    D[0] = dadd(suma, s2[0]);
    {
        dual buff = ddiv(dk(1.0), D[0]);
        for (int j = 0; j < Jt; j++) {
            dual arg = dmulc(d[j], t[0]);
            dual co = dcos(arg), si = dsin(arg);
            V[2 * j + 1] = dmul(buff, si);
            V[2 * j] = dmul(buff, co);
            U[2 * j + 1] = dsub(dmul(a[j], si), dmul(b[j], co));
            U[2 * j] = dadd(dmul(a[j], co), dmul(b[j], si));
        }
    }
    for (int64_t n = 1; n < N; n++) {
        dual s = dk(0.0);
        real tn = t[n], dt = tn - (real)t[n - 1];
        dual *Un = U + (size_t)R * n, *Vn = V + (size_t)R * n, *Vp = V + (size_t)R * (n - 1);
        dual *ph = phi + (size_t)R * (n - 1);
        for (int j = 0; j < Jt; j++) {
            dual arg = dmulc(d[j], tn);
            dual co = dcos(arg), si = dsin(arg), ec = dexp(dmulc(dneg(c[j]), dt));
            ph[2 * j + 1] = ec; ph[2 * j] = ec;
            Un[2 * j + 1] = dsub(dmul(a[j], si), dmul(b[j], co));
            Un[2 * j] = dadd(dmul(a[j], co), dmul(b[j], si));
            Vn[2 * j + 1] = si; Vn[2 * j] = co;
        }
        for (int j = 0; j < R; j++) {
            dual uj = Un[j], vn = Vp[j];
            dual phj = ph[j];
            dual dn = dmul(D[n - 1], vn);
            dual vnj = Vn[j];
            for (int k = 0; k < j; k++) {
                dual uk = Un[k];
                dual r = dmul(dadd(S[j + (size_t)k * R], dmul(dn, Vp[k])), dmul(phj, ph[k]));
                S[j + (size_t)k * R] = r;
                dual v = dmul(uj, r);
                Vn[k] = dsub(Vn[k], v);
                vnj = dsub(vnj, dmul(uk, r));
                s = dadd(s, dmul(dmulc(v, 2.0), uk));
            }
            S[j + (size_t)j * R] = dmul(dadd(S[j + (size_t)j * R], dmul(dn, vn)), dmul(phj, phj));
            dual r = dmul(S[j + (size_t)j * R], uj);
            s = dadd(s, dmul(r, uj));
            Vn[j] = dsub(vnj, r);
        }
        dual dn = dsub(dadd(suma, s2[n]), s);
        D[n] = dn;
        for (int j = 0; j < R; j++) Vn[j] = ddiv(Vn[j], dn);
    }
    {
        dual logdetD = dlog(D[0]);
        z[0] = y[0];
        for (int64_t n = 1; n < N; n++) {
            dual s = dk(0.0), zp = z[n - 1];
            const dual *Wp = V + (size_t)R * (n - 1), *Un = U + (size_t)R * n;
            const dual *ph = phi + (size_t)R * (n - 1);
            for (int j = 0; j < R; j++) {
                f[j] = dmul(dadd(f[j], dmul(Wp[j], zp)), ph[j]);
                s = dadd(s, dmul(Un[j], f[j]));
            }
            logdetD = dadd(logdetD, dlogabs(D[n]));
            z[n] = dsub(y[n], s);
        }
        z[N - 1] = ddiv(z[N - 1], D[N - 1]);
        for (int64_t n = N - 2; n >= 0; n--) {
            dual s = dk(0.0), zn = z[n + 1];
            const dual *Un1 = U + (size_t)R * (n + 1), *Wn = V + (size_t)R * n;
            const dual *ph = phi + (size_t)R * n;
            for (int j = 0; j < R; j++) {
                g[j] = dmul(dadd(g[j], dmul(Un1[j], zn)), ph[j]);
                s = dadd(s, dmul(Wn[j], g[j]));
            }
            z[n] = dsub(ddiv(z[n], D[n]), s);
        }
        dual yz = dk(0.0);
        for (int64_t n = 0; n < N; n++) yz = dadd(yz, dmul(y[n], z[n]));
        result = dsub(dsub(ddivc(dneg(logdetD), 2.0), dk((real)N * RM(log)(2 * R_PI) / 2)), ddivc(yz, 2.0));
    }
done:
    free(S); free(phi); free(U); free(V); free(D); free(z); free(f); free(g);
    return result;
}

/* One coefficient set with its data along one direction: (y − μ, ν s2) formed on duals. */
static dual logl_direction(int Jt, const dual *a, const dual *b, const dual *c, const dual *d, dual mu, dual nu, int64_t N,
                           const double *t, const double *y, const double *s2, const double *dy, const double *ds2,
                           dual *ybuf, dual *sbuf)
{
    for (int64_t n = 0; n < N; n++) {
        ybuf[n] = dsub(dmk(y[n], dy ? dy[n] : 0.0), mu);
        sbuf[n] = dmul(nu, dmk(s2[n], ds2 ? ds2[n] : 0.0));
    }
    return celerite_logl_jvp(Jt, a, b, c, d, N, t, ybuf, sbuf);
}

/* Shapes of pioran_celerite_logl_jvp (include/pioran_b200.h): a … d [B × Jt]; mu, nu [B] or NULL (0, 1); y_batch, s2_batch
 * [B × N] or NULL (then y, s2); tangents da … dd [B × P × Jt], dmu, dnu [B × P], dy, ds2 [B × P × N], each NULL = zero.
 * logl_out [B] or NULL, dlogl_out [B × P]. */
void ORC_JVP_ENTRY(int B, int Jt, int P, const double *a, const double *b, const double *c, const double *d, const double *mu,
                   const double *nu, int64_t N, const double *t, const double *y, const double *s2, const double *y_batch,
                   const double *s2_batch, const double *da, const double *db, const double *dc, const double *dd,
                   const double *dmu, const double *dnu, const double *dy, const double *ds2, double *logl_out, double *dlogl_out)
{
    dual *co = (dual *)malloc(sizeof(dual) * 4 * (size_t)Jt);
    dual *yb = (dual *)malloc(sizeof(dual) * (size_t)N);
    dual *sb = (dual *)malloc(sizeof(dual) * (size_t)N);
    if (!co || !yb || !sb) { free(co); free(yb); free(sb); return; }
    for (int i = 0; i < B; i++) {
        const double *yi = y_batch ? y_batch + (size_t)i * N : y, *si = s2_batch ? s2_batch + (size_t)i * N : s2;
        for (int p = 0; p < P; p++) {
            const size_t ip = (size_t)i * P + p, o = (size_t)i * Jt, to = ip * Jt;
            for (int m = 0; m < Jt; m++) {
                co[m] = dmk(a[o + m], da ? da[to + m] : 0.0);
                co[Jt + m] = dmk(b[o + m], db ? db[to + m] : 0.0);
                co[2 * Jt + m] = dmk(c[o + m], dc ? dc[to + m] : 0.0);
                co[3 * Jt + m] = dmk(d[o + m], dd ? dd[to + m] : 0.0);
            }
            dual mui = dmk(mu ? mu[i] : 0.0, dmu ? dmu[ip] : 0.0), nui = dmk(nu ? nu[i] : 1.0, dnu ? dnu[ip] : 0.0);
            dual L = logl_direction(Jt, co, co + Jt, co + 2 * Jt, co + 3 * Jt, mui, nui, N, t, yi, si,
                                    dy ? dy + ip * N : NULL, ds2 ? ds2 + ip * N : NULL, yb, sb);
            if (p == 0 && logl_out) logl_out[i] = (double)L.v;
            dlogl_out[ip] = (double)L.d;
        }
    }
    free(co); free(yb); free(sb);
}

/* ------------------------------------------------------------------------------------------------ approx with features on duals */
static dual psd_eval_dual(int model, const dual *p, real f)
{
    dual x = ddiv(dk(f), p[1]);
    dual v = ddiv(dpow(x, dneg(p[0])), dadd(dk(1.0), dpow(x, dsub(p[2], p[0]))));
    if (model == 1) v = ddiv(v, dadd(dk(1.0), dpow(ddiv(dk(f), p[3]), dsub(p[4], p[2]))));
    return v;
}

static int lu_solve_dual(int n, real *A, dual *x)
{
    for (int k = 0; k < n; k++) {
        int piv = k;
        real best = RM(fabs)(A[k + (size_t)k * n]);
        for (int i = k + 1; i < n; i++) {
            real v = RM(fabs)(A[i + (size_t)k * n]);
            if (v > best) { best = v; piv = i; }
        }
        if (best == 0.0) return -1;
        if (piv != k) {
            for (int j = 0; j < n; j++) {
                real tmp = A[k + (size_t)j * n];
                A[k + (size_t)j * n] = A[piv + (size_t)j * n];
                A[piv + (size_t)j * n] = tmp;
            }
            dual tmp = x[k]; x[k] = x[piv]; x[piv] = tmp;
        }
        real inv = 1.0 / A[k + (size_t)k * n];
        for (int i = k + 1; i < n; i++) A[i + (size_t)k * n] *= inv;
        for (int j = k + 1; j < n; j++) {
            real akj = A[k + (size_t)j * n];
            for (int i = k + 1; i < n; i++) A[i + (size_t)j * n] -= A[i + (size_t)k * n] * akj;
        }
    }
    for (int k = 0; k < n; k++)
        for (int i = k + 1; i < n; i++) x[i] = dsub(x[i], dmulc(x[k], A[i + (size_t)k * n]));
    for (int k = n - 1; k >= 0; k--) {
        x[k] = ddivc(x[k], A[k + (size_t)k * n]);
        for (int i = 0; i < k; i++) x[i] = dsub(x[i], dmulc(x[k], A[i + (size_t)k * n]));
    }
    return 0;
}

/* src/psd.jl:301-305, 318-324 (linear in the amplitudes) */
static dual integral_basis_dual(int J, const dual *a, const real *c, real x, int basis)
{
    dual acc = dk(0.0);
    if (basis == 0) {
        const real s2 = RM(sqrt)(2.0);
        for (int j = 0; j < J; j++) {
            real poly = (x * x + s2 * c[j] * x + c[j] * c[j]) / (x * x - s2 * c[j] * x + c[j] * c[j]);
            real br = RM(log)(poly) + 2.0 * RM(atan2)(c[j] * s2 * x, c[j] * c[j] - x * x);
            acc = dadd(acc, dmulc(ddivc(dmulc(a[j], c[j]), 4.0 * s2), br));
        }
    } else {
        const real s3 = RM(sqrt)(3.0);
        for (int j = 0; j < J; j++) {
            real drw = RM(atan)(x / c[j]);
            real poly = (x * x + s3 * c[j] * x + c[j] * c[j]) / (x * x - s3 * c[j] * x + c[j] * c[j]);
            real cel = 0.5 * RM(atan2)(x * x - c[j] * c[j], c[j] * x) + s3 / 4.0 * RM(log)(poly);
            acc = dadd(acc, dmulc(ddivc(dmulc(a[j], c[j]), 3.0), drw + cel));
        }
    }
    return acc;
}

/* src/psd.jl:330-334 integral_celerite on duals */
static dual integral_celerite_dual(dual a, dual b, dual c, dual d, real x)
{
    dual dp = dadd(d, dk(2.0 * R_PI * x)), dm = dsub(d, dk(2.0 * R_PI * x));
    dual num = dadd(dmul(c, c), dmul(dp, dp)), den = dadd(dmul(c, c), dmul(dm, dm));
    dual at = dsub(datan2(c, dm), datan2(c, dp));
    return ddivc(dadd(dmulc(dmul(a, at), 2.0), dmul(b, dlog(ddiv(num, den)))), 2.0 * R_PI);
}

/* orc_approx_features (oracle/pioran_oracle.c) on duals: continuum + nfeat QPO terms; returns the term count or < 0. */
static int approx_features_dual(int model, const dual *psd_par, real f_min, real f_max, int J, dual norm, real S_low, real S_high,
                                int is_integrated_power, int basis, int nfeat, const dual *feat, dual *a, dual *b, dual *c, dual *d)
{
    real f0 = f_min / S_low, fM = f_max * S_high;
    real *B = (real *)malloc(sizeof(real) * (size_t)J * J);
    real *fj = (real *)malloc(sizeof(real) * J);
    dual *amp = (dual *)malloc(sizeof(dual) * J);
    dual *cf = (dual *)malloc(sizeof(dual) * 4 * (nfeat > 0 ? nfeat : 1));
    double *Bd = (double *)malloc(sizeof(double) * (size_t)J * J);
    double *fd = (double *)malloc(sizeof(double) * J);
    int Jt = -2;
    if (!B || !fj || !amp || !cf || !Bd || !fd) goto out;
    orc_build_approx(J, (double)f0, (double)fM, basis, fd, Bd);
    for (int j = 0; j < J; j++) fj[j] = fd[j];
    for (size_t q = 0; q < (size_t)J * J; q++) B[q] = Bd[q];
    dual p0 = psd_eval_dual(model, psd_par, fj[0]);
    for (int j = 0; j < J; j++) amp[j] = ddiv(psd_eval_dual(model, psd_par, fj[j]), p0);
    if (lu_solve_dual(J, B, amp)) { Jt = -1; goto out; }
    for (int k = 0; k < nfeat; k++) {                          /* src/psd.jl:15-28 */
        dual S0 = feat[3 * k], fq = feat[3 * k + 1], Q = feat[3 * k + 2];
        dual Delta = dsqrt(dsub(dmulc(dmul(Q, Q), 4.0), dk(1.0)));
        dual w0 = dmulc(fq, 2.0 * R_PI);
        dual ak = ddivc(dmul(dmul(S0, w0), Q), 4.0);
        dual ck = ddivc(ddiv(w0, Q), 2.0);
        cf[4 * k] = ddiv(ak, p0); cf[4 * k + 1] = ddiv(ddiv(ak, Delta), p0); cf[4 * k + 2] = ck; cf[4 * k + 3] = dmul(ck, Delta);
    }
    dual integ;
    if (is_integrated_power) {
        integ = dsub(integral_basis_dual(J, amp, fj, f_max, basis), integral_basis_dual(J, amp, fj, f_min, basis));
        for (int k = 0; k < nfeat; k++)
            integ = dadd(integ, dsub(integral_celerite_dual(cf[4 * k], cf[4 * k + 1], cf[4 * k + 2], cf[4 * k + 3], f_max),
                                     integral_celerite_dual(cf[4 * k], cf[4 * k + 1], cf[4 * k + 2], cf[4 * k + 3], f_min)));
    } else {
        dual s = dk(0.0);
        for (int j = 0; j < J; j++) s = dadd(s, dmulc(amp[j], fj[j]));
        integ = (basis == 0) ? ddivc(dmulc(s, R_PI), RM(sqrt)(2.0)) : ddivc(dmulc(s, 2.0 * R_PI), 3.0);
    }
    dual scale = ddiv(norm, integ);
    for (int j = 0; j < J; j++) amp[j] = dmul(amp[j], scale);
    for (int k = 0; k < nfeat; k++) { cf[4 * k] = dmul(cf[4 * k], scale); cf[4 * k + 1] = dmul(cf[4 * k + 1], scale); }
    if (basis == 0) {
        for (int j = 0; j < J; j++) {
            a[j] = ddivc(dmulc(dmulc(amp[j], fj[j]), R_PI), RM(sqrt)(2.0)); b[j] = a[j];
            c[j] = dk(RM(sqrt)(2.0) * R_PI * fj[j]); d[j] = c[j];
        }
        Jt = J;
    } else {
        for (int j = 0; j < J; j++) {
            dual aj = ddivc(dmulc(dmulc(amp[j], fj[j]), R_PI), 3.0);
            real cj = R_PI * fj[j];
            a[j] = aj;     b[j] = dmulc(aj, RM(sqrt)(3.0)); c[j] = dk(cj);           d[j] = dk(RM(sqrt)(3.0) * cj);
            a[J + j] = aj; b[J + j] = dk(0.0);              c[J + j] = dk(2.0 * cj); d[J + j] = dk(0.0);
        }
        Jt = 2 * J;
    }
    for (int k = 0; k < nfeat; k++) {                          /* src/psd.jl:254-259, 277-282 */
        a[Jt + k] = dmulc(cf[4 * k], 2.0); b[Jt + k] = dmulc(cf[4 * k + 1], 2.0); c[Jt + k] = cf[4 * k + 2]; d[Jt + k] = cf[4 * k + 3];
    }
    Jt += nfeat;
out:
    free(B); free(fj); free(amp); free(cf); free(Bd); free(fd);
    return Jt;
}

/* Gradient of the likelihood with features: θ row = [psd parameters…, norm, ν, μ, (S₀, f₀, Q)…] (pioran_approx_features_logl);
 * one dual sweep per column.  logl_out [B] or NULL, grad_out [B × ncol]. */
void ORC_FEAT_ENTRY(int model, int n_psd_par, int nfeat, int B, const double *theta, double f_min, double f_max, int J,
                    double S_low, double S_high, int is_integrated_power, int basis, int64_t N, const double *t, const double *y,
                    const double *s2, double *logl_out, double *grad_out)
{
    const int ncol = n_psd_par + 3 + 3 * nfeat, Jmax = 2 * J + nfeat;
    dual *co = (dual *)malloc(sizeof(dual) * 4 * (size_t)Jmax);
    dual *yb = (dual *)malloc(sizeof(dual) * (size_t)N);
    dual *sb = (dual *)malloc(sizeof(dual) * (size_t)N);
    dual par[8], feat[3 * 8];
    if (!co || !yb || !sb || nfeat > 8) { free(co); free(yb); free(sb); return; }
    for (int i = 0; i < B; i++) {
        const double *th = theta + (size_t)i * ncol;
        for (int k = 0; k < ncol; k++) {
            for (int q = 0; q < n_psd_par; q++) par[q] = dmk(th[q], q == k ? 1.0 : 0.0);
            dual norm = dmk(th[n_psd_par], k == n_psd_par ? 1.0 : 0.0);
            dual nu = dmk(th[n_psd_par + 1], k == n_psd_par + 1 ? 1.0 : 0.0);
            dual mu = dmk(th[n_psd_par + 2], k == n_psd_par + 2 ? 1.0 : 0.0);
            for (int q = 0; q < 3 * nfeat; q++) feat[q] = dmk(th[n_psd_par + 3 + q], k == n_psd_par + 3 + q ? 1.0 : 0.0);
            int Jt = approx_features_dual(model, par, f_min, f_max, J, norm, S_low, S_high, is_integrated_power, basis, nfeat, feat,
                                          co, co + Jmax, co + 2 * Jmax, co + 3 * Jmax);
            dual L = Jt > 0 ? logl_direction(Jt, co, co + Jmax, co + 2 * Jmax, co + 3 * Jmax, mu, nu, N, t, y, s2, NULL, NULL, yb, sb)
                            : dmk(NAN, NAN);
            if (k == 0 && logl_out) logl_out[i] = (double)L.v;
            grad_out[(size_t)i * ncol + k] = (double)L.d;
        }
    }
    free(co); free(yb); free(sb);
}
