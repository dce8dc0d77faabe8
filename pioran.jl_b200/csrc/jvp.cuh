// jvp.cuh — K5g: Jacobian-vector product of the explicit-coefficient log-likelihood (FP64, sm_100a), ranks up to 96.
//
// ForwardDiff's chunk mode over logl(a, b, c, d, τ, y, σ²) (reference: test/test_likelihood.jl:55, and every NUTS model built on a
// `:celerite_gpu` solver): for parameter vector i and direction p the kernel returns ∂/∂ε of
//     logl(a_i + ε da_ip, b_i + ε db_ip, c_i + ε dc_ip, d_i + ε dd_ip, τ, ỹ_i, σ̃²_i),
//     ỹ_i = y_i + ε dy_ip − (μ_i + ε dμ_ip),   σ̃²_i = (ν_i + ε dν_ip)(s2_i + ε ds2_ip),
// and the value logL.  Unlike the approx-path gradients (grad.cuh, wide_grad.cuh), the decay rates c and frequencies d carry
// tangents too, so the row tables do: with θ_n = d t_n and Δ_n = t_n − t_{n−1},
//     complex term  U̇_cos = ȧ cos + ḃ sin + ḋ t_n (b cos − a sin)     U̇_sin = ȧ sin − ḃ cos + ḋ t_n (a cos + b sin)
//                   V̇ = ḋ t_n (−sin, cos)                               φ̇ = −ċ Δ_n φ
//     real term     U̇ = ȧ,  V̇ = 0,  φ̇ = −ċ Δ_n φ.
// Real terms (b = d = 0 for every parameter vector of the batch; make_term_rows in api.cu) take one row and IGNORE db, dd: this is
// exact, ∂k/∂b = e^{−c|τ|} sin(d|τ|) and ∂k/∂d = |τ| e^{−c|τ|}(b cos(dτ) − a sin(d|τ|)) vanish at b = d = 0.
//
// Layout: the register-file CTA of wide.cuh (celerite_wide_reg_kernel) on (value, tangent) pairs, as in wide_grad.cuh — one CTA
// of 256 threads per (parameter vector, direction), thread (ty, tx) of a 16×16 grid owning the interleaved TS×TS tile of the
// full-square state T and of its tangent Ṫ (TS = ⌈R/16⌉ = 1 … 6).  The value is recomputed in every CTA; the direction-0 CTA
// writes logL.  Per step, on top of the value recursion of wide.cuh:
//     Ṫ ← φ̇_r (φ_c T) + φ_r (φ̇_c T + φ_c Ṫ) + (q̇φ)_r (wφ)_c + (qφ)_r (ẇφ)_c,     (qφ)˙ = q̇ φ + q φ̇,  (wφ)˙ = ẇ φ + w φ̇
//     ṗ = Ṫ U + T U̇;   Ḋ = Σȧ + (νs2)˙ − U̇ᵀp − Uᵀṗ;   ż = ỹ̇ − U̇ᵀg − Uᵀġ;   ġ ← φ̇ (g + w z) + φ (ġ + ẇ z + w ż)
//     q̇ = V̇ − ṗ;   ẇ = (q̇ − w Ḋ) / D;   (log L)˙ = −½ Σ Ḋ/D − ½ Σ (2 z ż − z² Ḋ/D) / D.
// The step rule is prototyped and checked against central differences in tests/tools/proto/jvp_math.py.
#pragma once
#include "wide.cuh"

namespace pioran {

constexpr int JVP_MAX_RANK = 96;

struct JvpArgs {
    const double* t; const double* y; const double* s2;   // resident series [N]
    int64_t N;
    const double *a, *b, *c, *d;                           // [B × Jt]
    const double *mu, *nu;                                 // [B] or nullptr (0, 1)
    const double *y_batch, *s2_batch;                      // [B × N] or nullptr (the resident series)
    const double *da, *db, *dc, *dd;                       // [B × P × Jt] or nullptr (zero tangent)
    const double *dmu, *dnu;                               // [B × P] or nullptr
    const double *dy, *ds2;                                // [B × P × N] or nullptr
    const int* term_row;                                   // [Jt], as in the generic kernels
    int Jt, P;
    double* logl;                                          // [B] or nullptr
    double* dlogl;                                         // [B × P]
};

// grid = B · P; block = 256.
template <int TS>
__global__ void __launch_bounds__(WIDE_THREADS, 1) celerite_jvp_kernel(const JvpArgs args) {
    constexpr int LD = 16 * TS, NWARP = WIDE_THREADS / 32;
    __shared__ __align__(16) double tabU[WIDE_CH][LD], tabV[WIDE_CH][LD], tabP[WIDE_CH][LD];
    __shared__ __align__(16) double tabdU[WIDE_CH][LD], tabdV[WIDE_CH][LD], tabdP[WIDE_CH][LD];
    __shared__ __align__(16) double qphi[LD], wphi[LD], dqphi[LD], dwphi[LD], p_s[LD], dp_s[LD];
    __shared__ double red[4 * NWARP];
    __shared__ double sums[3];   // Σa, Σȧ, D_0: read in phase 3 instead of held in registers

    const int P = args.P, Jt = args.Jt;
    const int i = blockIdx.x / P, k = blockIdx.x - i * P;
    const size_t ik = (size_t)i * P + k;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ty = tid >> 4, tx = tid & 15;
    const int64_t N = args.N;
    const double* t = args.t;
    // inputs are read from the kernel parameters where they are used, not held in registers across the sweep: at TS = 6 the
    // two tiles take nearly all of them
    const size_t cjo = (size_t)i * Jt, tjo = ik * Jt;

    if (tid == 0) {
        double suma = 0.0, dsuma = 0.0;
        for (int m = 0; m < Jt; m++) { suma += args.a[cjo + m]; if (args.da) dsuma += args.da[tjo + m]; }   // celerite_solver.jl:21
        sums[0] = suma; sums[1] = dsuma; sums[2] = 1.0;
    }

    double Tm[TS][TS], dT[TS][TS];
#pragma unroll
    for (int r = 0; r < TS; r++)
#pragma unroll
        for (int j = 0; j < TS; j++) { Tm[r][j] = 0.0; dT[r][j] = 0.0; }
    for (int q = tid; q < WIDE_CH * LD; q += WIDE_THREADS) {
        (&tabU[0][0])[q] = 0.0; (&tabV[0][0])[q] = 0.0; (&tabP[0][0])[q] = 0.0;
        (&tabdU[0][0])[q] = 0.0; (&tabdV[0][0])[q] = 0.0; (&tabdP[0][0])[q] = 0.0;
    }
    const bool owner = tid < LD;
    double g = 0.0, dg = 0.0, q = 0.0, dq = 0.0, w = 0.0, dw = 0.0, zprev = 0.0, dzprev = 0.0;
    double chi2 = 0.0, dchi2 = 0.0, dlog = 0.0;
    double logacc = 0.0, dkeep = 1.0;
    const bool b3 = (tx & 8) != 0, b2 = (tx & 4) != 0, b1 = (tx & 2) != 0;
    __syncthreads();

    for (int64_t nb = 0; nb < N; nb += WIDE_CH) {
        const int ns = (int)((N - nb) < WIDE_CH ? (N - nb) : WIDE_CH);
        // ---- U, V, φ of the next ns steps and their tangents (celerite_solver.jl:51-64), one thread per (step, term)
        for (int idx = tid; idx < ns * Jt; idx += WIDE_THREADS) {
            const int s = idx / Jt, m = idx - s * Jt;
            const int64_t n = nb + s;
            const double tn = t[n];
            const double dt_n = (n >= 1) ? tn - t[n - 1] : 0.0;
            const double ph = (n >= 1) ? exp(-args.c[cjo + m] * dt_n) : 0.0;
            const double dph = args.dc ? -args.dc[tjo + m] * dt_n * ph : 0.0;
            const double am = args.a[cjo + m], dam = args.da ? args.da[tjo + m] : 0.0;
            const int tr = args.term_row[m];
            if (tr < 0) {     // real term: one row, U = a, V = 1
                const int r0 = -tr - 1;
                tabU[s][r0] = am; tabV[s][r0] = 1.0; tabP[s][r0] = ph;
                tabdU[s][r0] = dam; tabdV[s][r0] = 0.0; tabdP[s][r0] = dph;
            } else {
                double si, co;
                sincos_large(args.d[cjo + m] * tn, &si, &co);
                const double bm = args.b[cjo + m], dbm = args.db ? args.db[tjo + m] : 0.0, dtd = args.dd ? args.dd[tjo + m] * tn : 0.0;
                const double uc = am * co + bm * si, us = am * si - bm * co;
                tabU[s][tr] = uc;                 // celerite_solver.jl:60
                tabU[s][tr + 1] = us;             // celerite_solver.jl:59
                tabV[s][tr] = co; tabV[s][tr + 1] = si;
                tabP[s][tr] = ph; tabP[s][tr + 1] = ph;
                tabdU[s][tr] = fma(dam, co, fma(dbm, si, -dtd * us));
                tabdU[s][tr + 1] = fma(dam, si, fma(-dbm, co, dtd * uc));
                tabdV[s][tr] = -dtd * si; tabdV[s][tr + 1] = dtd * co;
                tabdP[s][tr] = dph; tabdP[s][tr + 1] = dph;
            }
        }
        __syncthreads();
        for (int s = 0; s < ns; s++) {
            const int64_t n = nb + s;
            const double* Un = tabU[s];
            const double* Vn = tabV[s];
            const double* Pn = tabP[s];
            const double* dUn = tabdU[s];
            const double* dPn = tabdP[s];
            // ---- phase 0: owners publish (q, w)φ and their tangents, advance g, ġ
            if (owner) {
                const double ph = Pn[tid], dph = dPn[tid];
                qphi[tid] = q * ph; wphi[tid] = w * ph;
                dqphi[tid] = fma(dq, ph, q * dph); dwphi[tid] = fma(dw, ph, w * dph);
                const double gin = fma(w, zprev, g);
                dg = fma(dph, gin, ph * fma(dw, zprev, fma(w, dzprev, dg)));
                g = ph * gin;                              // celerite_solver.jl:137
            }
            __syncthreads();
            // ---- phase 1: tile update and row sums, value and tangent
            // at TS = 6 the row-side tangents φ̇_r, (q̇φ)_r are read from shared memory where they are used: held in registers
            // next to the two 6×6 tiles they would spill
            constexpr bool DPH_REG = TS < 6;
            double phr[TS], dphr[DPH_REG ? TS : 1], qr[TS], dqr[DPH_REG ? TS : 1], rs[8], drs[8];
#pragma unroll
            for (int r = 0; r < TS; r++) {
                const int ridx = ty + 16 * r;
                phr[r] = Pn[ridx]; qr[r] = qphi[ridx];
                if (DPH_REG) { dphr[DPH_REG ? r : 0] = dPn[ridx]; dqr[DPH_REG ? r : 0] = dqphi[ridx]; }
            }
#pragma unroll
            for (int r = 0; r < 8; r++) { rs[r] = 0.0; drs[r] = 0.0; }
#pragma unroll
            for (int j = 0; j < TS; j++) {
                const int cidx = tx + 16 * j;
                const double pc = Pn[cidx], dpc = dPn[cidx], wc = wphi[cidx], dwc = dwphi[cidx], uc = Un[cidx], duc = dUn[cidx];
#pragma unroll
                for (int r = 0; r < TS; r++) {
                    const double aT = pc * Tm[r][j];
                    const double t1 = fma(phr[r], aT, qr[r] * wc);                                // celerite_solver.jl:76
                    // volatile: a plain load would be hoisted out of the column loop into the registers it is meant to spare
                    const double dph_r = DPH_REG ? dphr[DPH_REG ? r : 0] : static_cast<const volatile double*>(dPn)[ty + 16 * r];
                    const double dq_r = DPH_REG ? dqr[DPH_REG ? r : 0] : static_cast<const volatile double*>(dqphi)[ty + 16 * r];
                    const double dt1 = fma(dph_r, aT, fma(phr[r], fma(dpc, Tm[r][j], pc * dT[r][j]), fma(dq_r, wc, qr[r] * dwc)));
                    Tm[r][j] = t1; dT[r][j] = dt1;
                    rs[r] = fma(t1, uc, rs[r]);
                    drs[r] = fma(dt1, uc, fma(t1, duc, drs[r]));
                }
            }
            {   // reduce-scatter of the (padded) 8 row sums over the 16 lanes that share ty, both components
                double e4[4], e2[2], f4[4], f2[2];
#pragma unroll
                for (int m = 0; m < 4; m++) {
                    const double r0 = __shfl_xor_sync(FULL, b3 ? rs[m] : rs[m + 4], 8);
                    const double r1 = __shfl_xor_sync(FULL, b3 ? drs[m] : drs[m + 4], 8);
                    e4[m] = (b3 ? rs[m + 4] : rs[m]) + r0;
                    f4[m] = (b3 ? drs[m + 4] : drs[m]) + r1;
                }
#pragma unroll
                for (int m = 0; m < 2; m++) {
                    const double r0 = __shfl_xor_sync(FULL, b2 ? e4[m] : e4[m + 2], 4);
                    const double r1 = __shfl_xor_sync(FULL, b2 ? f4[m] : f4[m + 2], 4);
                    e2[m] = (b2 ? e4[m + 2] : e4[m]) + r0;
                    f2[m] = (b2 ? f4[m + 2] : f4[m]) + r1;
                }
                const double r0 = __shfl_xor_sync(FULL, b1 ? e2[0] : e2[1], 2);
                const double r1 = __shfl_xor_sync(FULL, b1 ? f2[0] : f2[1], 2);
                double tot = (b1 ? e2[1] : e2[0]) + r0;
                double dtot = (b1 ? f2[1] : f2[0]) + r1;
                tot += __shfl_xor_sync(FULL, tot, 1);
                dtot += __shfl_xor_sync(FULL, dtot, 1);
                const int isel = 4 * (b3 ? 1 : 0) + 2 * (b2 ? 1 : 0) + (b1 ? 1 : 0);
                if ((tx & 1) == 0 && isel < TS) { p_s[ty + 16 * isel] = tot; dp_s[ty + 16 * isel] = dtot; }
            }
            __syncthreads();
            // ---- phase 2: UᵀTU, Uᵀg and their tangents
            double p = 0.0, dp = 0.0, v4[4] = {0.0, 0.0, 0.0, 0.0};
            if (owner) {
                p = p_s[tid]; dp = dp_s[tid];
                const double u = Un[tid], du = dUn[tid];
                v4[0] = u * p;
                v4[1] = fma(du, p, u * dp);
                v4[2] = u * g;
                v4[3] = fma(du, g, u * dg);
            }
#pragma unroll
            for (int sft = 16; sft >= 1; sft >>= 1)
#pragma unroll
                for (int m = 0; m < 4; m++) v4[m] += __shfl_xor_sync(FULL, v4[m], sft);
            if (lane == 0)
#pragma unroll
                for (int m = 0; m < 4; m++) red[4 * warp + m] = v4[m];
            __syncthreads();
            double t4[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int wq = 0; wq < NWARP; wq++)
#pragma unroll
                for (int m = 0; m < 4; m++) t4[m] += red[4 * wq + m];
            // ---- phase 3: pivot, innovation, next q and w — on pairs
            const double mu = args.mu ? args.mu[i] : 0.0, nu = args.nu ? args.nu[i] : 1.0;
            const double dmu = args.dmu ? args.dmu[ik] : 0.0, dnu = args.dnu ? args.dnu[ik] : 0.0;
            const double s2n = args.s2_batch ? args.s2_batch[(size_t)i * N + n] : args.s2[n];
            const double yn = args.y_batch ? args.y_batch[(size_t)i * N + n] : args.y[n];
            const double ds2n = args.ds2 ? args.ds2[ik * N + n] : 0.0;
            const double D = fma(nu, s2n, sums[0]) - t4[0];                          // celerite_solver.jl:92
            const double dD = fma(dnu, s2n, fma(nu, ds2n, sums[1])) - t4[1];
            const double z = (yn - mu) - t4[2];                                // celerite_solver.jl:141
            const double dz = ((args.dy ? args.dy[ik * N + n] : 0.0) - dmu) - t4[3];
            const double rD = 1.0 / D;
            if (owner) {
                q = Vn[tid] - p; dq = tabdV[s][tid] - dp;                         // celerite_solver.jl:95-98 (W = q / D)
                w = q * rD;
                dw = (dq - w * dD) * rD;
            }
            zprev = z; dzprev = dz;
            chi2 = fma(z * z, rD, chi2);
            dchi2 = fma(fma(2.0 * z, dz, -(z * z) * (dD * rD)), rD, dchi2);
            dlog = fma(dD, rD, dlog);
            if (warp == NWARP - 1) {                                             // celerite_solver.jl:126,140
                if (n == 0) { if (lane == 0) sums[2] = D; }
                else if ((int)(n & 31) == lane) dkeep = D;
                if ((n & 31) == 31) { logacc += log(fabs(dkeep)); dkeep = 1.0; }
            }
        }
        __syncthreads();   // the tables are rebuilt for the next WIDE_CH steps
    }
    if (warp == NWARP - 1) {
        double la = logacc + log(fabs(dkeep));
#pragma unroll
        for (int sft = 16; sft >= 1; sft >>= 1) la += __shfl_xor_sync(FULL, la, sft);
        const double logdet = log(sums[2]) + la;                                  // no abs on the first pivot (celerite_solver.jl:126)
        if (lane == 0) {
            if (k == 0 && args.logl) args.logl[i] = -logdet / 2 - (double)N * 1.8378770664093453 / 2 - chi2 / 2;   // celerite_solver.jl:333
            args.dlogl[ik] = -dlog / 2 - dchi2 / 2;
        }
    }
}

}  // namespace pioran
