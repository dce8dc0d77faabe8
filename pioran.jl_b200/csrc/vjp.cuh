// vjp.cuh — K5r: vector-Jacobian product (reverse mode) of the explicit-coefficient log-likelihood (FP64, sm_100a), ranks up to 96.
//
// For coefficient set i the kernel returns logL_i and, in one backward sweep, ∂logL_i with respect to a, b, c, d [Jt], μ_i, ν_i and
// the data row as it enters (y, s2 [N]; ỹ = y − μ, σ̃² = ν·s2, the conventions of K5g's dy / ds2 tangents).  It differentiates the
// same function as K5g (jvp.cuh): log|D_n| has derivative 1/D_n whatever the sign of D_n, NaN and Inf propagate as data, and a
// real term (b = d = 0 for every set of the batch, one row) reports ∂/∂b = ∂/∂d = 0 exactly.
//
// The adjoint step rule (state adjoint T̄ kept symmetric, so every contraction is a row sum of the tile) is written out in
// tests/tools/proto/vjp_math.py and checked there by duality, <gradient, v> = forward-mode derivative along v.
//
// Layout: the register-file CTA of K5g without tangents — one CTA of 256 threads per set, thread (ty, tx) owning the interleaved
// TS×TS tile of T (forward) and of T̄ (backward), TS = ⌈R/16⌉ = 1 … 6.  Three passes over the series:
//   1. forward: the value sweep of wide.cuh; writes q_n, g_n [R] and D_n, z_n once per step, and checkpoints the tile T_{n−1} at
//      every n ≡ 0 (mod K) (K ≈ √N, a multiple of WIDE_CH);
//   2. per segment [s0, s0 + K), last first: restore the checkpoint and replay the tile recursion T ← (φφᵀ)∘(T + q wᵀ) from the
//      stored q, D (no reductions), writing T_{n−1} of every step of the segment;
//   3. backward over the segment: the adjoint step, reading T_{n−1} and the per-step values once each.
// Workspace per set: vjp_ws_doubles(TS, N, K) doubles; the host bounds it by processing the batch in θ-chunks.
#pragma once
#include "wide.cuh"

namespace pioran {

constexpr int VJP_MAX_RANK = 96;

struct VjpArgs {
    const double* t; const double* y; const double* s2;   // resident series [N]
    int64_t N;
    const double *a, *b, *c, *d;                           // [B × Jt]
    const double *mu, *nu;                                 // [B] or nullptr (0, 1)
    const double *y_batch, *s2_batch;                      // [B × N] or nullptr (the resident series)
    const int* term_row;                                   // [Jt], as in the generic kernels
    int Jt, K;                                             // K: steps per checkpoint segment, a multiple of WIDE_CH
    double* ws;                                            // [B × vjp_ws_doubles(TS, N, K)]
    double* logl;                                          // [B] or nullptr
    double *ga, *gb, *gc, *gd;                             // [B × Jt] or nullptr
    double *gmu, *gnu;                                     // [B] or nullptr
    double *gy, *gs2;                                      // [B × N] or nullptr
};

// Per set, in doubles: q_n, g_n [N × 16·TS], D_n, z_n [N], ⌈N/K⌉ checkpoint tiles and K segment tiles of 256·TS² doubles each
// (thread-fastest, so every tile store and load is coalesced).
__host__ __device__ inline size_t vjp_ws_doubles(int TS, int64_t N, int K) {
    const size_t LD = 16 * (size_t)TS, tile = (size_t)WIDE_THREADS * TS * TS;
    return (size_t)N * (2 * LD + 2) + ((size_t)((N + K - 1) / K) + (size_t)K) * tile;
}

// -DPIORAN_VJP_CHECKS: in-kernel checks of the workspace indexing (a debug build; off in the library)
#ifdef PIORAN_VJP_CHECKS
#include <cassert>
#define VJP_CHECK(cond) assert(cond)
#else
#define VJP_CHECK(cond) ((void)0)
#endif

// U, V, φ of steps nb … nb + ns − 1 (celerite_solver.jl:51-64), one thread per (step, term); padded rows stay zero.
template <int LD>
__device__ __forceinline__ void vjp_tables(const VjpArgs& args, size_t cjo, int64_t nb, int ns, double (*tabU)[LD], double (*tabV)[LD],
                                           double (*tabP)[LD]) {
    for (int idx = threadIdx.x; idx < ns * args.Jt; idx += WIDE_THREADS) {
        const int s = idx / args.Jt, m = idx - s * args.Jt;
        const int64_t n = nb + s;
        const double tn = args.t[n];
        const double ph = (n >= 1) ? exp(-args.c[cjo + m] * (tn - args.t[n - 1])) : 0.0;
        const double am = args.a[cjo + m];
        const int tr = args.term_row[m];
        if (tr < 0) {
            const int r0 = -tr - 1;
            tabU[s][r0] = am; tabV[s][r0] = 1.0; tabP[s][r0] = ph;
        } else {
            double si, co;
            sincos_large(args.d[cjo + m] * tn, &si, &co);
            const double bm = args.b[cjo + m];
            tabU[s][tr] = am * co + bm * si; tabU[s][tr + 1] = am * si - bm * co;
            tabV[s][tr] = co; tabV[s][tr + 1] = si;
            tabP[s][tr] = ph; tabP[s][tr + 1] = ph;
        }
    }
}

// Sum of the (padded) 8 row sums rs over the 16 lanes that share ty; the even lane tx = 2·isel ends with row sum isel.
__device__ __forceinline__ double vjp_rowsum(const double (&rs)[8], bool b3, bool b2, bool b1) {
    double e4[4], e2[2];
#pragma unroll
    for (int m = 0; m < 4; m++) e4[m] = (b3 ? rs[m + 4] : rs[m]) + __shfl_xor_sync(FULL, b3 ? rs[m] : rs[m + 4], 8);
#pragma unroll
    for (int m = 0; m < 2; m++) e2[m] = (b2 ? e4[m + 2] : e4[m]) + __shfl_xor_sync(FULL, b2 ? e4[m] : e4[m + 2], 4);
    double tot = (b1 ? e2[1] : e2[0]) + __shfl_xor_sync(FULL, b1 ? e2[0] : e2[1], 2);
    return tot + __shfl_xor_sync(FULL, tot, 1);
}

// grid = B; block = 256.
template <int TS>
__global__ void __launch_bounds__(WIDE_THREADS, 1) celerite_vjp_kernel(const VjpArgs args) {
    constexpr int LD = 16 * TS, NWARP = WIDE_THREADS / 32, TT = TS * TS;
    __shared__ __align__(16) double tabU[WIDE_CH][LD], tabV[WIDE_CH][LD], tabP[WIDE_CH][LD], tabQ[WIDE_CH][LD], tabW[WIDE_CH][LD];
    __shared__ __align__(16) double vA[LD], vB[LD], vC[LD], rsum[4][LD];
    __shared__ double red[2 * NWARP];
    __shared__ double sums[3];   // Σa, D_0, Σ D̄
    __shared__ int rkind[LD];    // 0 padding, 1 real row, 2 cos row, 3 sin row

    const int i = blockIdx.x, Jt = args.Jt, K = args.K;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ty = tid >> 4, tx = tid & 15;
    const int64_t N = args.N;
    const size_t cjo = (size_t)i * Jt;
    const bool owner = tid < LD;
    const bool b3 = (tx & 8) != 0, b2 = (tx & 4) != 0, b1 = (tx & 2) != 0;
    const int isel = 4 * (b3 ? 1 : 0) + 2 * (b2 ? 1 : 0) + (b1 ? 1 : 0);
    const bool writer = (tx & 1) == 0 && isel < TS;
    const int64_t nseg = (N + K - 1) / K;
    const size_t stride = vjp_ws_doubles(TS, N, K);
    double* const wsq = args.ws + (size_t)i * stride;
    double* const wsg = wsq + (size_t)N * LD;
    double* const wsD = wsg + (size_t)N * LD;
    double* const wsz = wsD + N;
    double* const ck = wsz + N;
    double* const seg = ck + (size_t)nseg * TT * WIDE_THREADS;
    VJP_CHECK(seg + (size_t)K * TT * WIDE_THREADS == wsq + stride && K % WIDE_CH == 0);
    const double mu = args.mu ? args.mu[i] : 0.0, nu = args.nu ? args.nu[i] : 1.0;

    if (tid == 0) {
        double suma = 0.0;
        for (int m = 0; m < Jt; m++) suma += args.a[cjo + m];   // celerite_solver.jl:21
        sums[0] = suma; sums[1] = 1.0;
    }
    for (int q = tid; q < WIDE_CH * LD; q += WIDE_THREADS) {
        (&tabU[0][0])[q] = 0.0; (&tabV[0][0])[q] = 0.0; (&tabP[0][0])[q] = 0.0; (&tabQ[0][0])[q] = 0.0; (&tabW[0][0])[q] = 0.0;
    }
    if (owner) rkind[tid] = 0;
    __syncthreads();
    for (int m = tid; m < Jt; m += WIDE_THREADS) {
        const int tr = args.term_row[m];
        if (tr < 0) rkind[-tr - 1] = 1;
        else { rkind[tr] = 2; rkind[tr + 1] = 3; }
    }

    // ================================================================ pass 1: forward value sweep, per-step values, checkpoints
    double Tm[TS][TS];
#pragma unroll
    for (int r = 0; r < TS; r++)
#pragma unroll
        for (int j = 0; j < TS; j++) Tm[r][j] = 0.0;
    double g = 0.0, q = 0.0, w = 0.0, zprev = 0.0, chi2 = 0.0, logacc = 0.0, dkeep = 1.0;
    __syncthreads();
    for (int64_t nb = 0; nb < N; nb += WIDE_CH) {
        const int ns = (int)((N - nb) < WIDE_CH ? (N - nb) : WIDE_CH);
        vjp_tables<LD>(args, cjo, nb, ns, tabU, tabV, tabP);
        __syncthreads();
        for (int s = 0; s < ns; s++) {
            const int64_t n = nb + s;
            if (n % K == 0) {   // checkpoint T_{n−1}
                double* dst = ck + (size_t)(n / K) * TT * WIDE_THREADS + tid;
                VJP_CHECK(n / K < nseg);
#pragma unroll
                for (int r = 0; r < TS; r++)
#pragma unroll
                    for (int j = 0; j < TS; j++) dst[(r * TS + j) * WIDE_THREADS] = Tm[r][j];
            }
            if (owner) {
                const double ph = tabP[s][tid];
                vA[tid] = q * ph; vB[tid] = w * ph;
                g = ph * fma(w, zprev, g);                // celerite_solver.jl:137
                wsg[(size_t)n * LD + tid] = g;
            }
            __syncthreads();
            double phr[TS], qr[TS], rs[8];
#pragma unroll
            for (int r = 0; r < TS; r++) { phr[r] = tabP[s][ty + 16 * r]; qr[r] = vA[ty + 16 * r]; }
#pragma unroll
            for (int r = 0; r < 8; r++) rs[r] = 0.0;
#pragma unroll
            for (int j = 0; j < TS; j++) {
                const int cidx = tx + 16 * j;
                const double pc = tabP[s][cidx], wc = vB[cidx], uc = tabU[s][cidx];
#pragma unroll
                for (int r = 0; r < TS; r++) {
                    const double t1 = fma(phr[r], pc * Tm[r][j], qr[r] * wc);   // celerite_solver.jl:76
                    Tm[r][j] = t1;
                    rs[r] = fma(t1, uc, rs[r]);
                }
            }
            const double tot = vjp_rowsum(rs, b3, b2, b1);
            if (writer) rsum[0][ty + 16 * isel] = tot;
            __syncthreads();
            double p = 0.0, v0 = 0.0, v1 = 0.0;
            if (owner) {
                p = rsum[0][tid];
                const double u = tabU[s][tid];
                v0 = u * p; v1 = u * g;
            }
#pragma unroll
            for (int sft = 16; sft >= 1; sft >>= 1) { v0 += __shfl_xor_sync(FULL, v0, sft); v1 += __shfl_xor_sync(FULL, v1, sft); }
            if (lane == 0) { red[2 * warp] = v0; red[2 * warp + 1] = v1; }
            __syncthreads();
            double t0 = 0.0, t1 = 0.0;
#pragma unroll
            for (int wq = 0; wq < NWARP; wq++) { t0 += red[2 * wq]; t1 += red[2 * wq + 1]; }
            const double s2n = args.s2_batch ? args.s2_batch[(size_t)i * N + n] : args.s2[n];
            const double yn = args.y_batch ? args.y_batch[(size_t)i * N + n] : args.y[n];
            const double D = fma(nu, s2n, sums[0]) - t0;                       // celerite_solver.jl:92
            const double z = (yn - mu) - t1;                                   // celerite_solver.jl:141
            const double rD = 1.0 / D;
            if (owner) {
                q = tabV[s][tid] - p;                                          // celerite_solver.jl:95-98 (W = q / D)
                w = q * rD;
                wsq[(size_t)n * LD + tid] = q;
            }
            if (tid == 0) { wsD[n] = D; wsz[n] = z; }
            zprev = z;
            chi2 = fma(z * z, rD, chi2);
            if (warp == NWARP - 1) {                                           // celerite_solver.jl:126,140
                if (n == 0) { if (lane == 0) sums[1] = D; }
                else if ((int)(n & 31) == lane) dkeep = D;
                if ((n & 31) == 31) { logacc += log(fabs(dkeep)); dkeep = 1.0; }
            }
        }
        __syncthreads();
    }
    if (warp == NWARP - 1) {
        double la = logacc + log(fabs(dkeep));
#pragma unroll
        for (int sft = 16; sft >= 1; sft >>= 1) la += __shfl_xor_sync(FULL, la, sft);
        const double logdet = log(sums[1]) + la;                                  // no abs on the first pivot (celerite_solver.jl:126)
        if (lane == 0 && args.logl) args.logl[i] = -logdet / 2 - (double)N * 1.8378770664093453 / 2 - chi2 / 2;   // celerite_solver.jl:333
    }

    // ================================================================ passes 2 and 3, segment by segment from the end
    double Tb[TS][TS];
#pragma unroll
    for (int r = 0; r < TS; r++)
#pragma unroll
        for (int j = 0; j < TS; j++) Tb[r][j] = 0.0;
    double qb = 0.0, wb = 0.0, gb = 0.0;                    // owners: q̄_n, w̄_n, ḡ_n as left by step n + 1
    double acca = 0.0, accb = 0.0, accc = 0.0, accd = 0.0;  // owners: the row's share of its term's ā, b̄, c̄, d̄
    double sD = 0.0, sDs2 = 0.0, sz = 0.0;                  // Σ D̄, Σ D̄ s2, Σ z̄ (every thread; thread 0 writes them)
    double qc = 0.0, gcur = 0.0;                            // owners: q_n, g_n of the step being reversed
    double Dc = wsD[N - 1], zc = wsz[N - 1];
    if (owner) { qc = wsq[(size_t)(N - 1) * LD + tid]; gcur = wsg[(size_t)(N - 1) * LD + tid]; }
    for (int64_t sg = nseg - 1; sg >= 0; sg--) {
        const int64_t s0 = sg * K, s1 = (s0 + K < N) ? s0 + K : N;
        {   // ---- pass 2: T_{n−1} of every step of the segment, from its checkpoint
            const double* src = ck + (size_t)sg * TT * WIDE_THREADS + tid;
#pragma unroll
            for (int r = 0; r < TS; r++)
#pragma unroll
                for (int j = 0; j < TS; j++) Tm[r][j] = src[(r * TS + j) * WIDE_THREADS];
        }
        for (int64_t nb = s0; nb < s1; nb += WIDE_CH) {
            const int ns = (int)((s1 - nb) < WIDE_CH ? (s1 - nb) : WIDE_CH);
            vjp_tables<LD>(args, cjo, nb, ns, tabU, tabV, tabP);
            __syncthreads();
            for (int idx = tid; idx < ns * LD; idx += WIDE_THREADS) {   // (qφ), (wφ) as the forward pass formed them
                const int s = idx / LD, r = idx - s * LD;
                const int64_t n = nb + s;
                double qv = 0.0, wv = 0.0;
                if (n >= 1) { qv = wsq[(size_t)(n - 1) * LD + r]; wv = qv * (1.0 / wsD[n - 1]); }
                tabQ[s][r] = qv * tabP[s][r]; tabW[s][r] = wv * tabP[s][r];
            }
            __syncthreads();
            for (int s = 0; s < ns; s++) {
                const int64_t n = nb + s;
                double* dst = seg + (size_t)(n - s0) * TT * WIDE_THREADS + tid;
                VJP_CHECK(n - s0 < K);
#pragma unroll
                for (int r = 0; r < TS; r++)
#pragma unroll
                    for (int j = 0; j < TS; j++) dst[(r * TS + j) * WIDE_THREADS] = Tm[r][j];
                if (n + 1 < s1) {
#pragma unroll
                    for (int j = 0; j < TS; j++) {
                        const int cidx = tx + 16 * j;
                        const double pc = tabP[s][cidx], wc = tabW[s][cidx];
#pragma unroll
                        for (int r = 0; r < TS; r++) Tm[r][j] = fma(tabP[s][ty + 16 * r], pc * Tm[r][j], tabQ[s][ty + 16 * r] * wc);
                    }
                }
            }
            __syncthreads();
        }
        // ---- pass 3: the adjoint steps of the segment, last first
        for (int64_t nb = s0 + ((s1 - 1 - s0) / WIDE_CH) * WIDE_CH; nb >= s0; nb -= WIDE_CH) {
            const int ns = (int)((s1 - nb) < WIDE_CH ? (s1 - nb) : WIDE_CH);
            vjp_tables<LD>(args, cjo, nb, ns, tabU, tabV, tabP);
            __syncthreads();
            for (int s = ns - 1; s >= 0; s--) {
                const int64_t n = nb + s;
                double qp = 0.0, gp = 0.0, Dp = 1.0, zp = 0.0;   // step n − 1 (zero before the first step)
                if (n >= 1) {
                    if (owner) { qp = wsq[(size_t)(n - 1) * LD + tid]; gp = wsg[(size_t)(n - 1) * LD + tid]; }
                    Dp = wsD[n - 1]; zp = wsz[n - 1];
                }
                const double rD = 1.0 / Dc, wcur = qc * rD, wp = qp * (1.0 / Dp);
                // ---- phase A: z̄, D̄ (two dot products over the rows), then p̄ and the row-local adjoints
                double v0 = wb * wcur, v1 = gb * wcur;
#pragma unroll
                for (int sft = 16; sft >= 1; sft >>= 1) { v0 += __shfl_xor_sync(FULL, v0, sft); v1 += __shfl_xor_sync(FULL, v1, sft); }
                if (lane == 0) { red[2 * warp] = v0; red[2 * warp + 1] = v1; }
                __syncthreads();
                double sww = 0.0, sgw = 0.0;
#pragma unroll
                for (int wq = 0; wq < NWARP; wq++) { sww += red[2 * wq]; sgw += red[2 * wq + 1]; }
                const double zr = zc * rD;
                const double zbar = sgw - zr;
                const double Dbar = fma(0.5 * zr, zr, -0.5 * rD) - sww * rD;
                double ub = 0.0, qbn = 0.0, gbn = 0.0;
                if (owner) {
                    const double u = tabU[s][tid];
                    qbn = fma(wb, rD, qb);
                    gbn = fma(-zbar, u, gb);
                    ub = -zbar * gcur - Dbar * (tabV[s][tid] - qc);
                    vA[tid] = fma(-Dbar, u, -qbn);   // p̄
                    vB[tid] = qp; vC[tid] = wp;
                }
                __syncthreads();
                // ---- phase B: T̄ update and its four row sums: T_n p̄, (T̄∘Tin) φ, T̄ w_{n−1}, T̄ q_{n−1}
                {
                    const double* src = seg + (size_t)(n - s0) * TT * WIDE_THREADS + tid;
                    // at TS >= 5 the row-side u and q_{n−1} are read from shared memory where they are used: held in registers
                    // next to T̄ and the four row-sum arrays they would spill
                    constexpr bool ROW_REG = TS < 5;
                    double phr[TS], pbr[TS], ur[ROW_REG ? TS : 1], qmr[ROW_REG ? TS : 1], rs0[8], rs1[8], rs2[8], rs3[8];
#pragma unroll
                    for (int r = 0; r < TS; r++) {
                        const int ridx = ty + 16 * r;
                        phr[r] = tabP[s][ridx]; pbr[r] = vA[ridx];
                        if (ROW_REG) { ur[ROW_REG ? r : 0] = tabU[s][ridx]; qmr[ROW_REG ? r : 0] = vB[ridx]; }
                    }
#pragma unroll
                    for (int r = 0; r < 8; r++) { rs0[r] = 0.0; rs1[r] = 0.0; rs2[r] = 0.0; rs3[r] = 0.0; }
#pragma unroll
                    for (int j = 0; j < TS; j++) {
                        const int cidx = tx + 16 * j;
                        const double pc = tabP[s][cidx], pbc = vA[cidx], uc = tabU[s][cidx], qmc = vB[cidx], wmc = vC[cidx];
#pragma unroll
                        for (int r = 0; r < TS; r++) {
                            // volatile: a plain load would be hoisted out of the column loop into the registers it is meant to spare
                            const double u_r = ROW_REG ? ur[ROW_REG ? r : 0] : static_cast<const volatile double*>(&tabU[s][0])[ty + 16 * r];
                            const double qm_r = ROW_REG ? qmr[ROW_REG ? r : 0] : static_cast<const volatile double*>(vB)[ty + 16 * r];
                            const double tp = src[(r * TS + j) * WIDE_THREADS];            // T_{n−1}
                            const double tin = fma(qm_r, wmc, tp);
                            const double tn = fma(phr[r], pc * tp, (qm_r * phr[r]) * (wmc * pc));
                            rs0[r] = fma(tn, pbc, rs0[r]);
                            double tb = fma(0.5, fma(pbr[r], uc, u_r * pbc), Tb[r][j]);
                            rs1[r] = fma(tb * tin, pc, rs1[r]);
                            tb = phr[r] * (pc * tb);
                            Tb[r][j] = tb;
                            rs2[r] = fma(tb, wmc, rs2[r]);
                            rs3[r] = fma(tb, qmc, rs3[r]);
                        }
                    }
                    const double o0 = vjp_rowsum(rs0, b3, b2, b1), o1 = vjp_rowsum(rs1, b3, b2, b1);
                    const double o2 = vjp_rowsum(rs2, b3, b2, b1), o3 = vjp_rowsum(rs3, b3, b2, b1);
                    if (writer) {
                        const int ridx = ty + 16 * isel;
                        rsum[0][ridx] = o0; rsum[1][ridx] = o1; rsum[2][ridx] = o2; rsum[3][ridx] = o3;
                    }
                }
                __syncthreads();
                // ---- phase C: φ̄, the row tables' adjoints mapped to the terms, and the state adjoints of step n − 1
                if (owner) {
                    ub += rsum[0][tid];
                    const double ph = tabP[s][tid];
                    const double phb = fma(2.0, rsum[1][tid], gbn * fma(wp, zp, gp));
                    const double tn = args.t[n], dtn = n >= 1 ? tn - args.t[n - 1] : 0.0;
                    accc = fma(-dtn * ph, phb, accc);
                    const int kind = rkind[tid];
                    if (kind == 1) {
                        acca += ub;
                    } else if (kind == 2) {
                        const double co = tabV[s][tid], si = tabV[s][tid + 1], us = tabU[s][tid + 1];
                        acca = fma(ub, co, acca); accb = fma(ub, si, accb); accd = fma(tn, -(ub * us) - qbn * si, accd);
                    } else if (kind == 3) {
                        const double co = tabV[s][tid - 1], si = tabV[s][tid], uc = tabU[s][tid - 1];
                        acca = fma(ub, si, acca); accb = fma(-ub, co, accb); accd = fma(tn, fma(ub, uc, qbn * co), accd);
                    }
                    const double ginb = ph * gbn;
                    qb = rsum[2][tid];
                    wb = fma(ginb, zp, rsum[3][tid]);
                    gb = ginb;
                }
                const double s2n = args.s2_batch ? args.s2_batch[(size_t)i * N + n] : args.s2[n];
                sD += Dbar; sDs2 = fma(Dbar, s2n, sDs2); sz += zbar;
                if (tid == 0) {
                    if (args.gy) args.gy[(size_t)i * N + n] = zbar;
                    if (args.gs2) args.gs2[(size_t)i * N + n] = nu * Dbar;
                }
                qc = qp; gcur = gp; Dc = Dp; zc = zp;
            }
            __syncthreads();   // the tables are rebuilt for the previous WIDE_CH steps
        }
    }
    // ---- per-row shares → per-term gradients
    if (owner) { rsum[0][tid] = acca; rsum[1][tid] = accb; rsum[2][tid] = accc; rsum[3][tid] = accd; }
    if (tid == 0) {
        sums[2] = sD;
        if (args.gmu) args.gmu[i] = -sz;
        if (args.gnu) args.gnu[i] = sDs2;
    }
    __syncthreads();
    for (int m = tid; m < Jt; m += WIDE_THREADS) {
        const int tr = args.term_row[m];
        double gav, gbv = 0.0, gcv, gdv = 0.0;
        if (tr < 0) {
            const int r0 = -tr - 1;
            gav = rsum[0][r0]; gcv = rsum[2][r0];
        } else {
            gav = rsum[0][tr] + rsum[0][tr + 1]; gbv = rsum[1][tr] + rsum[1][tr + 1];
            gcv = rsum[2][tr] + rsum[2][tr + 1]; gdv = rsum[3][tr] + rsum[3][tr + 1];
        }
        if (args.ga) args.ga[cjo + m] = gav + sums[2];
        if (args.gb) args.gb[cjo + m] = gbv;
        if (args.gc) args.gc[cjo + m] = gcv;
        if (args.gd) args.gd[cjo + m] = gdv;
    }
}

// ∂logL/∂θ_p = Σ_m (ā ȧ + b̄ ḃ + c̄ ċ + d̄ ḋ)_{m,p} + μ̄ μ̇_p + ν̄ ν̇_p: the K5r gradients contracted with the coefficient tangents
// along every θ column, in the layout approx_features_grad_kernel writes (tangents [B × P × Jt], [B × P]).  One thread per (i, p).
__global__ void vjp_contract_kernel(int B, int P, int Jt, const double* ga, const double* gb, const double* gc, const double* gd,
                                    const double* gmu, const double* gnu, const double* da, const double* db, const double* dc,
                                    const double* dd, const double* dmu, const double* dnu, double* out) {
    const size_t ip = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ip >= (size_t)B * P) return;
    const size_t i = ip / P, co = i * Jt, to = ip * Jt;
    double acc = fma(gmu[i], dmu[ip], gnu[i] * dnu[ip]);
    for (int m = 0; m < Jt; m++)
        acc = fma(ga[co + m], da[to + m], fma(gb[co + m], db[to + m], fma(gc[co + m], dc[to + m], fma(gd[co + m], dd[to + m], acc))));
    out[ip] = acc;
}

}  // namespace pioran
