// postvar.cuh — K6: posterior predictive variance of the celerite GP (the diagonal of `predict_cov`,
// src/direct_solver.jl:28-119, behind var / std of a PosteriorGP, src/scalable_GP.jl:44-155) in O((N + M)·R²) per parameter
// vector, from the factor (W_n, D_n) that the STEP_STORE sweep of the posterior mean leaves in HBM.  No matrix inverse.
//
//   var(τ) = k(0) − k(τ, t)ᵀ K̃⁻¹ k(τ, t) = D_τ − g_τᵀ Ξ_{n₀} g_τ      (n₀ = #{t_n < τ}, K̃ = K + diag(ν σ²))
//
// (a) forward replay: Q_n = (φ_n φ_nᵀ) ∘ Q_{n−1} + D_n W_n W_nᵀ (the state just after absorbing point n; a decay and a
//     rank-1 update per step, no reductions).  A prediction point in gap n₀ sees S_τ = (e_τ e_τᵀ) ∘ Q_{n₀−1} (e_τ: row decay
//     t_{n₀−1} → τ) and stores into the workspace
//         D_τ = Σa − U(τ)ᵀ S_τ U(τ)              the filter variance from the data before τ
//         g_τ = e_{τ→t_{n₀}} ∘ (S_τ U(τ) − V(τ))  the seed of the forward substitution of k(τ, ·) over the data after τ;
// (b) backward sweep of the "future information matrix" Ξ_n = U_n U_nᵀ / D_n + A_nᵀ X A_n, A_n = I − W_n U_nᵀ,
//     X = (φ_{n+1} φ_{n+1}ᵀ) ∘ Ξ_{n+1}, applied as a rank-2 update
//         p = X W_n,  s = W_nᵀ p,  Ξ_n = X − U_n pᵀ − p U_nᵀ + (s + 1/D_n) U_n U_nᵀ,
//     and at each gap var(τ) = D_τ − g_τᵀ Ξ_{n₀} g_τ.  The numpy restatement is tests/tools/proto/postvar_math.py.
//
// Layout: one CTA of 256 threads per parameter vector, the register-file tile of celerite_wide_reg_kernel (wide.cuh):
// thread (ty, tx) of a 16×16 grid owns rows {ty + 16·i} × columns {tx + 16·j}, i, j < TS = ⌈R/16⌉, of the full square
// (Q and Ξ are symmetric; keeping both triangles makes every contraction a row sum).  U, W, φ and D of WIDE_PV_CH steps are
// staged in shared memory; rows R … 16·TS − 1 are zero.  cos/sin are taken at absolute times (sincos_large, common.cuh).
// A parameter vector whose factor has a pivot D_n ≤ 0 (or NaN) gets NaN in every entry of its row.
//
// COV = true (the first launch of the posterior covariance, postcov.cuh) also writes, per prediction point, the two vectors
// the covariance walk K8 reads:  r(τ) = S_τ U(τ) − V(τ) (pass 1, before the decay to t_{n₀}) and the start vector
// w₀(τ) = U(τ) + e_{τ→t_{n₀}} ∘ (Ξ_{n₀} g_τ) (U(τ) in pass 1, the Ξ term in pass 2); a bad pivot makes both NaN.
// COV = false compiles to the variance kernel alone.
#pragma once
#include <type_traits>
#include "common.cuh"
#include "wide.cuh"

namespace pioran {

constexpr int PV_CH = 8;   // steps whose U, W, φ, D are staged at once

struct PostVarArgs {
    const double* t; const double* tau;   // data times [N], prediction times [M] (ascending)
    const int* n0;                        // [M] number of data times strictly below τ_m
    int64_t N; int64_t M;
    int Jt, R, RPL;                       // rank, leading dimension of the stored factor
    const double* a; const double* b; const double* c; const double* d;   // [B × Jt]
    const int* term_row;                  // as in the generic K2 kernel
    const double* W; const double* D;     // stored factor [B × N × RPL], [B × N]
    double* ws;                           // workspace [B × M × (R + 1)]: g_τ (R entries), then D_τ
    double* var;                          // [B × M]
};
struct PostVarCovArgs : PostVarArgs {     // COV = true: the variance kernel's arguments and
    double* pt;                           // [B × M × 2R], r(τ) (R entries), then w₀(τ)
};

// Sum over the CTA of one value per thread, into slot `red` (8 doubles); the caller synchronises before reading it.
__device__ __forceinline__ void pv_block_part(double v, double* red, int lane, int warp) {
#pragma unroll
    for (int sft = 16; sft >= 1; sft >>= 1) v += __shfl_xor_sync(FULL, v, sft);
    if (lane == 0) red[warp] = v;
}

// Reduce-scatter of the (padded) 8 row sums over the 16 lanes that share ty (as in celerite_wide_reg_kernel): row
// ty + 16·i ends in `out[ty + 16·i]`.
template <int TS>
__device__ __forceinline__ void pv_row_sums(double (&rs)[8], double* out, int ty, int tx) {
    const bool b3 = (tx & 8) != 0, b2 = (tx & 4) != 0, b1 = (tx & 2) != 0;
    double e4[4], e2[2];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const double recv = __shfl_xor_sync(FULL, b3 ? rs[k] : rs[k + 4], 8);
        e4[k] = (b3 ? rs[k + 4] : rs[k]) + recv;
    }
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const double recv = __shfl_xor_sync(FULL, b2 ? e4[k] : e4[k + 2], 4);
        e2[k] = (b2 ? e4[k + 2] : e4[k]) + recv;
    }
    const double recv = __shfl_xor_sync(FULL, b1 ? e2[0] : e2[1], 2);
    double tot = (b1 ? e2[1] : e2[0]) + recv;
    tot += __shfl_xor_sync(FULL, tot, 1);
    const int isel = 4 * (b3 ? 1 : 0) + 2 * (b2 ? 1 : 0) + (b1 ? 1 : 0);
    if ((tx & 1) == 0 && isel < TS) out[ty + 16 * isel] = tot;
}

// grid = B (one CTA per parameter vector), block = WIDE_THREADS
template <int TS, bool COV = false>
__global__ void __launch_bounds__(WIDE_THREADS, TS <= 6 ? 2 : 1)
celerite_postvar_kernel(const typename std::conditional<COV, PostVarCovArgs, PostVarArgs>::type pa) {
    constexpr int LD = 16 * TS, NWARP = WIDE_THREADS / 32;
    __shared__ __align__(16) double tabU[PV_CH][LD], tabW[PV_CH][LD], tabP[PV_CH][LD];
    __shared__ double tabD[PV_CH];
    __shared__ __align__(16) double xs[LD], ys[2][LD];
    __shared__ double red[2][NWARP];
    __shared__ int rterm[LD], rkind[LD];   // row → term, ROW_COS / ROW_SIN / ROW_REAL / ROW_PAD

    const int th = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ty = tid >> 4, tx = tid & 15;
    const int Jt = pa.Jt, R = pa.R;
    const int64_t N = pa.N, M = pa.M;
    const double* ca = pa.a + (size_t)th * Jt;
    const double* cb = pa.b + (size_t)th * Jt;
    const double* cc = pa.c + (size_t)th * Jt;
    const double* cd = pa.d + (size_t)th * Jt;
    const double* Wg = pa.W + (size_t)th * N * pa.RPL;
    const double* Dg = pa.D + (size_t)th * N;
    const int LDG = R + 1;
    double* ws = pa.ws + (size_t)th * M * LDG;
    double* var = pa.var + (size_t)th * M;

    // a non-positive (or NaN) pivot: the factor does not exist, the whole row is NaN
    int bad = 0;
    for (int64_t n = tid; n < N; n += WIDE_THREADS) bad |= !(Dg[n] > 0.0);
    if (__syncthreads_or(bad)) {
        for (int64_t m = tid; m < M; m += WIDE_THREADS) var[m] = __longlong_as_double(0x7ff8000000000000LL);
        if constexpr (COV)
            for (int64_t k = tid; k < M * 2 * R; k += WIDE_THREADS)
                pa.pt[(size_t)th * M * 2 * R + k] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    for (int r = tid; r < LD; r += WIDE_THREADS) { rterm[r] = 0; rkind[r] = ROW_PAD; }
    __syncthreads();
    for (int m = tid; m < Jt; m += WIDE_THREADS) {
        const int tr = pa.term_row[m];
        if (tr < 0) { rterm[-tr - 1] = m; rkind[-tr - 1] = ROW_REAL; }
        else { rterm[tr] = m; rkind[tr] = ROW_COS; rterm[tr + 1] = m; rkind[tr + 1] = ROW_SIN; }
    }
    double suma = 0.0;
    for (int m = 0; m < Jt; m++) suma += ca[m];   // celerite_solver.jl:21

    double Tm[TS][TS];
#pragma unroll
    for (int i = 0; i < TS; i++)
#pragma unroll
        for (int j = 0; j < TS; j++) Tm[i][j] = 0.0;
    __syncthreads();

    // row r of U(x), V(x) for an owner thread (rows ≥ R are zero)
    auto row_uv = [&](int r, double x, double& u, double& v) {
        const int kind = rkind[r], m = rterm[r];
        if (kind == ROW_REAL) { u = ca[m]; v = 1.0; return; }
        if (kind == ROW_PAD) { u = 0.0; v = 0.0; return; }
        double si, co;
        sincos_large(cd[m] * x, &si, &co);
        if (kind == ROW_COS) { u = ca[m] * co + cb[m] * si; v = co; }   // celerite_solver.jl:60, 62
        else                 { u = ca[m] * si - cb[m] * co; v = si; }   // celerite_solver.jl:59, 63
    };

    // ================================================================ (a) forward replay
    // at gap n the tile holds Q_{n−1}; every prediction point of the gap reads it, then step n is absorbed
    int64_t mp = 0;
    auto forward_gap = [&](int64_t n) {
        for (; mp < M && pa.n0[mp] == n; mp++) {
            const double tm = pa.tau[mp];
            double e = 0.0, e2 = 0.0, v = 0.0;
            if (tid < LD) {
                double u;
                row_uv(tid, tm, u, v);
                if constexpr (COV)
                    if (tid < R) pa.pt[((size_t)th * M + mp) * 2 * R + R + tid] = u;   // w₀ = U(τ); pass 2 adds the Ξ term
                const double cr = rkind[tid] == ROW_PAD ? 0.0 : cc[rterm[tid]];
                e = n > 0 ? exp(-cr * (tm - pa.t[n - 1])) : 0.0;
                e2 = n < N ? exp(-cr * (pa.t[n] - tm)) : 0.0;
                xs[tid] = e * u;
            }
            __syncthreads();
            double rs[8], xr[TS];
#pragma unroll
            for (int i = 0; i < 8; i++) rs[i] = 0.0;
#pragma unroll
            for (int i = 0; i < TS; i++) xr[i] = xs[ty + 16 * i];
#pragma unroll
            for (int j = 0; j < TS; j++) {
                const double xc = xs[tx + 16 * j];
#pragma unroll
                for (int i = 0; i < TS; i++) rs[i] = fma(Tm[i][j], xc, rs[i]);
            }
            double quad = 0.0;   // xᵀ Q x
#pragma unroll
            for (int i = 0; i < TS; i++) quad = fma(xr[i], rs[i], quad);
            pv_block_part(quad, red[0], lane, warp);
            pv_row_sums<TS>(rs, ys[0], ty, tx);
            __syncthreads();
            if (tid < R) ws[mp * LDG + tid] = e2 * fma(e, ys[0][tid], -v);
            if constexpr (COV)
                if (tid < R) pa.pt[((size_t)th * M + mp) * 2 * R + tid] = fma(e, ys[0][tid], -v);   // r(τ)
            if (tid == 0) {
                double q = 0.0;
#pragma unroll
                for (int k = 0; k < NWARP; k++) q += red[0][k];
                ws[mp * LDG + R] = suma - q;
            }
        }
    };
    for (int64_t nb = 0; nb < N; nb += PV_CH) {
        const int ns = (int)((N - nb) < PV_CH ? (N - nb) : PV_CH);
        for (int idx = tid; idx < ns * LD; idx += WIDE_THREADS) {
            const int s = idx / LD, r = idx - s * LD;
            const int64_t n = nb + s;
            const bool on = r < R;
            tabW[s][r] = on ? Wg[n * pa.RPL + r] : 0.0;
            tabP[s][r] = (on && n >= 1) ? exp(-cc[rterm[r]] * (pa.t[n] - pa.t[n - 1])) : 0.0;
            if (r == 0) tabD[s] = Dg[n];
        }
        __syncthreads();
        for (int s = 0; s < ns; s++) {
            const int64_t n = nb + s;
            forward_gap(n);
            const double Dn = tabD[s];
            double phr[TS], dwr[TS];
#pragma unroll
            for (int i = 0; i < TS; i++) { phr[i] = tabP[s][ty + 16 * i]; dwr[i] = Dn * tabW[s][ty + 16 * i]; }
#pragma unroll
            for (int j = 0; j < TS; j++) {
                const double pc = tabP[s][tx + 16 * j], wc = tabW[s][tx + 16 * j];
#pragma unroll
                for (int i = 0; i < TS; i++) Tm[i][j] = fma(phr[i] * pc, Tm[i][j], dwr[i] * wc);   // (φφᵀ)∘Q + D w wᵀ
            }
        }
        __syncthreads();   // the tables are rebuilt for the next PV_CH steps
    }
    forward_gap(N);
    __syncthreads();       // the workspace rows of this CTA are read back below

    // ================================================================ (b) backward sweep of Ξ
    for (int64_t m = M - 1 - tid; m >= 0 && pa.n0[m] == N; m -= WIDE_THREADS) var[m] = ws[m * LDG + R];   // Ξ_N = 0
    mp = M - 1;
    while (mp >= 0 && pa.n0[mp] == N) mp--;
#pragma unroll
    for (int i = 0; i < TS; i++)
#pragma unroll
        for (int j = 0; j < TS; j++) Tm[i][j] = 0.0;
    int slot = 0;          // double-buffered reduction slots: no barrier between a read and the next write
    for (int64_t hi = N; hi > 0; hi -= PV_CH) {
        const int64_t lo = hi - PV_CH > 0 ? hi - PV_CH : 0;
        const int ns = (int)(hi - lo);
        for (int idx = tid; idx < ns * LD; idx += WIDE_THREADS) {
            const int s = idx / LD, r = idx - s * LD;
            const int64_t n = lo + s;
            const bool on = r < R;
            double u = 0.0, v;
            if (on) row_uv(r, pa.t[n], u, v);
            tabU[s][r] = u;
            tabW[s][r] = on ? Wg[n * pa.RPL + r] : 0.0;
            tabP[s][r] = (on && n + 1 < N) ? exp(-cc[rterm[r]] * (pa.t[n + 1] - pa.t[n])) : 0.0;
            if (r == 0) tabD[s] = Dg[n];
        }
        __syncthreads();
        for (int s = ns - 1; s >= 0; s--) {
            const int64_t n = lo + s;
            // ---- X = (φφᵀ) ∘ Ξ_{n+1};  p = X W_n (row sums), s = W_nᵀ p
            double rs[8], phr[TS], wr[TS];
#pragma unroll
            for (int i = 0; i < 8; i++) rs[i] = 0.0;
#pragma unroll
            for (int i = 0; i < TS; i++) { phr[i] = tabP[s][ty + 16 * i]; wr[i] = tabW[s][ty + 16 * i]; }
#pragma unroll
            for (int j = 0; j < TS; j++) {
                const double pc = tabP[s][tx + 16 * j], wc = tabW[s][tx + 16 * j];
#pragma unroll
                for (int i = 0; i < TS; i++) {
                    const double x = (phr[i] * pc) * Tm[i][j];
                    Tm[i][j] = x;
                    rs[i] = fma(x, wc, rs[i]);
                }
            }
            double quad = 0.0;
#pragma unroll
            for (int i = 0; i < TS; i++) quad = fma(wr[i], rs[i], quad);
            pv_block_part(quad, red[slot], lane, warp);
            pv_row_sums<TS>(rs, ys[slot], ty, tx);
            __syncthreads();
            // ---- Ξ_n = X + U (κ U − p)ᵀ − p Uᵀ,  κ = s + 1/D_n
            double sw = 0.0;
#pragma unroll
            for (int k = 0; k < NWARP; k++) sw += red[slot][k];
            const double kap = sw + 1.0 / tabD[s];
            double ur[TS], pr[TS];
#pragma unroll
            for (int i = 0; i < TS; i++) { ur[i] = tabU[s][ty + 16 * i]; pr[i] = ys[slot][ty + 16 * i]; }
#pragma unroll
            for (int j = 0; j < TS; j++) {
                const double uc = tabU[s][tx + 16 * j], pc = ys[slot][tx + 16 * j];
                const double hc = fma(kap, uc, -pc);
#pragma unroll
                for (int i = 0; i < TS; i++) Tm[i][j] = fma(ur[i], hc, fma(-pr[i], uc, Tm[i][j]));
            }
            slot ^= 1;
            // ---- prediction points of gap n: var = D_τ − g_τᵀ Ξ_n g_τ
            for (; mp >= 0 && pa.n0[mp] == n; mp--) {
                const double* g = ws + mp * LDG;
                double gr[TS], part = 0.0;
#pragma unroll
                for (int i = 0; i < TS; i++) gr[i] = ty + 16 * i < R ? g[ty + 16 * i] : 0.0;
#pragma unroll
                for (int j = 0; j < TS; j++) {
                    const double gc = tx + 16 * j < R ? g[tx + 16 * j] : 0.0;
                    double acc = 0.0;
#pragma unroll
                    for (int i = 0; i < TS; i++) acc = fma(Tm[i][j], gr[i], acc);
                    part = fma(acc, gc, part);
                }
                pv_block_part(part, red[slot], lane, warp);
                if constexpr (COV) {   // Ξ_n g_τ as row sums (Ξ is symmetric), into the start vector w₀
                    double rs[8];
#pragma unroll
                    for (int i = 0; i < 8; i++) rs[i] = 0.0;
#pragma unroll
                    for (int j = 0; j < TS; j++) {
                        const double gc = tx + 16 * j < R ? g[tx + 16 * j] : 0.0;
#pragma unroll
                        for (int i = 0; i < TS; i++) rs[i] = fma(Tm[i][j], gc, rs[i]);
                    }
                    pv_row_sums<TS>(rs, ys[slot], ty, tx);
                }
                __syncthreads();
                if constexpr (COV)
                    if (tid < R) {
                        const double e2 = exp(-cc[rterm[tid]] * (pa.t[n] - pa.tau[mp]));
                        double* w0 = pa.pt + ((size_t)th * M + mp) * 2 * R + R;
                        w0[tid] = fma(e2, ys[slot][tid], w0[tid]);
                    }
                if (tid == 0) {
                    double q = 0.0;
#pragma unroll
                    for (int k = 0; k < NWARP; k++) q += red[slot][k];
                    var[mp] = g[R] - q;
                }
                slot ^= 1;
            }
        }
        __syncthreads();   // the tables are rebuilt for the next PV_CH steps
    }
}

}  // namespace pioran
